"""ctypes binding of libb200ssm.so (include/b200_ssm.h).

The library is the product: there is NO CPU or PyTorch fallback.  If the shared object is missing
and cannot be built (nvcc absent), importing an op raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200ssm.so")

i32, u32, i64, f32 = C.c_int32, C.c_uint32, C.c_int64, C.c_float
vp = C.c_void_p


class SScanFwdParams(C.Structure):
    """b200_sscan_fwd_params (include/b200_ssm.h)."""
    _fields_ = [
        ("batch", i32), ("dim", i32), ("seqlen", i32), ("dstate", i32), ("n_groups", i32),
        ("io_dtype", i32), ("delta_softplus", i32), ("rev_mask", u32), ("u_group_div", i32), ("ckpt_every", i32),
        ("u_batch_stride", i64), ("u_group_stride", i64), ("u_row_stride", i64),
        ("delta_batch_stride", i64), ("delta_group_stride", i64), ("delta_row_stride", i64),
        ("B_batch_stride", i64), ("B_group_stride", i64), ("B_state_stride", i64),
        ("C_batch_stride", i64), ("C_group_stride", i64), ("C_state_stride", i64),
        ("z_batch_stride", i64), ("z_row_stride", i64),
        ("out_batch_stride", i64), ("out_row_stride", i64),
        ("u", vp), ("delta", vp), ("A", vp), ("B", vp), ("C", vp), ("D", vp), ("z", vp), ("delta_bias", vp),
        ("out", vp), ("last_state", vp), ("ckpt", vp),
    ]


class SScanBwdParams(C.Structure):
    """b200_sscan_bwd_params."""
    _fields_ = [
        ("f", SScanFwdParams),
        ("dout_batch_stride", i64), ("dout_group_stride", i64), ("dout_row_stride", i64), ("dout_group_div", i64),
        ("du_batch_stride", i64), ("du_row_stride", i64),
        ("ddelta_batch_stride", i64), ("ddelta_group_stride", i64), ("ddelta_row_stride", i64),
        ("dB_batch_stride", i64), ("dB_group_stride", i64), ("dB_state_stride", i64),
        ("dC_batch_stride", i64), ("dC_group_stride", i64), ("dC_state_stride", i64),
        ("dz_batch_stride", i64), ("dz_row_stride", i64),
        ("dout", vp), ("du", vp), ("ddelta", vp), ("dz", vp),
        ("dA", vp), ("dB", vp), ("dC", vp), ("dD", vp), ("ddelta_bias", vp),
    ]


class SsdFwdParams(C.Structure):
    """b200_ssd_fwd_params."""
    _fields_ = [
        ("batch", i32), ("seqlen", i32), ("nheads", i32), ("headdim", i32), ("n_groups", i32), ("dstate", i32),
        ("chunk_size", i32), ("io_dtype", i32), ("dt_softplus", i32), ("precision", i32),
        ("dt_min", f32), ("dt_max", f32),
        ("x_stride", i64 * 4), ("dt_stride", i64 * 3), ("B_stride", i64 * 4), ("C_stride", i64 * 4),
        ("out_stride", i64 * 4),
        ("x", vp), ("dt", vp), ("A", vp), ("B", vp), ("C", vp), ("D", vp), ("dt_bias", vp),
        ("initial_states", vp), ("out", vp), ("final_states", vp), ("workspace", vp),
        ("seq_idx", vp), ("seq_idx_stride", i64 * 2),
    ]


class SsdBwdParams(C.Structure):
    """b200_ssd_bwd_params."""
    _fields_ = [
        ("f", SsdFwdParams),
        ("dout_stride", i64 * 4),
        ("dout", vp), ("dx", vp), ("ddt", vp), ("dB", vp), ("dC", vp), ("dA", vp), ("dD", vp),
        ("ddt_bias", vp), ("scratch", vp),
        ("dx_stride", i64 * 4), ("ddt_stride", i64 * 3), ("dB_stride", i64 * 4), ("dC_stride", i64 * 4),
        ("final_states", vp), ("dfinal_states", vp), ("dinitial_states", vp),
    ]


class SsuParams(C.Structure):
    """b200_ssu_params."""
    _fields_ = [
        ("batch", i32), ("nheads", i32), ("headdim", i32), ("ngroups", i32), ("dstate", i32), ("dt_softplus", i32),
        ("state_dtype", i32), ("x_dtype", i32), ("dt_dtype", i32), ("A_dtype", i32), ("B_dtype", i32), ("C_dtype", i32),
        ("D_dtype", i32), ("z_dtype", i32), ("dt_bias_dtype", i32), ("out_dtype", i32),
        ("state_stride", i64 * 4), ("x_stride", i64 * 3), ("dt_stride", i64 * 3), ("A_stride", i64 * 3), ("B_stride", i64 * 3),
        ("C_stride", i64 * 3), ("D_stride", i64 * 2), ("z_stride", i64 * 3), ("dt_bias_stride", i64 * 2), ("out_stride", i64 * 3),
        ("state", vp), ("x", vp), ("dt", vp), ("A", vp), ("B", vp), ("C", vp), ("D", vp), ("z", vp), ("dt_bias", vp), ("out", vp),
    ]


_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}

# name -> (restype, argtypes) of every function include/b200_ssm.h declares, in the header's order
# (tests/test_abi.py parses the header and checks each entry)
SIGNATURES = {
    "b200_sscan_ckpt_bytes": (C.c_size_t, [i32] * 6),
    "b200_sscan_fwd": (C.c_int, [C.POINTER(SScanFwdParams), vp]),
    "b200_sscan_bwd": (C.c_int, [C.POINTER(SScanBwdParams), vp]),
    "b200_sscan_last_variant": (C.c_int, []),
    "b200_cross_scan_pack_strided": (C.c_int, [vp, vp, i64, i64, i64, i32, i32, i32, i32, vp]),
    "b200_cross_scan_unpack4": (C.c_int, [vp, vp, i64, i64, i64, vp, i32, i32, i32, i32, vp]),
    "b200_atrous_scan": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200_atrous_merge": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200_cross_scan_pack": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200_cross_scan_pack_bwd": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200_cross_merge": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200_cross_merge_bwd": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200_cross_scan4": (C.c_int, [vp, i64, vp, i32, i32, i32, i32, vp]),
    "b200_cross_scan4_bwd": (C.c_int, [vp, vp, i64, i32, i32, i32, i32, vp]),
    "b200_ssd_merge4": (C.c_int, [vp, vp, i32, i32, i32, i32, vp]),
    "b200_ssd_merge4_bwd": (C.c_int, [vp, vp, i32, i32, i32, i32, vp]),
    "b200_ssd_workspace_bytes": (C.c_size_t, [i32] * 7),
    "b200_ssd_bwd_scratch_bytes": (C.c_size_t, [i32] * 7),
    "b200_ssd_fwd": (C.c_int, [C.POINTER(SsdFwdParams), vp]),
    "b200_ssd_bwd": (C.c_int, [C.POINTER(SsdBwdParams), vp]),
    "b200_ssd_varlen_states": (C.c_int, [C.POINTER(SsdFwdParams), vp, i32, vp, vp]),
    "b200_rmsnorm_gated_fwd": (C.c_int, [vp, vp, vp, vp, vp, i64, i32, f32, vp]),
    "b200_rmsnorm_gated_bwd": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, i32, vp]),
    "b200_rmsnorm_grid": (C.c_int, [i64, i32, i32]),
    "b200_rmsnorm_fwd": (C.c_int, [vp, i32, i64, vp, i32, i64, vp, vp, vp, i32, vp, i64, i32, i32, i32, f32, vp]),
    "b200_rmsnorm_bwd": (C.c_int, [vp, i32, i64, vp, i32, i64, vp, i32, i64, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, vp]),
    "b200_ln_gate_grid": (C.c_int, [i64]),
    "b200_ln_gate_fwd": (C.c_int, [vp, i32, i64, vp, i64, i32, vp, vp, vp, i32, vp, vp, i64, i32, f32, vp]),
    "b200_ln_gate_bwd": (C.c_int, [vp, vp, i32, i64, vp, i64, i32, vp, vp, i32, vp, vp, vp, vp, vp, vp, i64, i32, vp]),
    "b200_dwconv_silu_fwd": (C.c_int, [vp, i64, i32, vp, vp, vp, i32, i32, i32, i32, vp]),
    "b200_dwconv_silu_bwd": (C.c_int, [vp, vp, i64, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    "b200_shuffle_cat_add_fwd": (C.c_int, [vp, i32, vp, i32, vp, vp, i32, i32, i32, i32, vp]),
    "b200_shuffle_cat_add_bwd": (C.c_int, [vp, i32, vp, i32, vp, i32, i32, i32, i32, vp]),
    "b200_patch_merge": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200_causal_conv1d_partials": (C.c_int, [i32] * 4),
    "b200_causal_conv1d_fwd": (C.c_int, [vp, i32, i64, i64, vp, vp, vp, i64, i64, vp, i32, i64, i64, i32, i32, i32, i32, i32, vp]),
    "b200_causal_conv1d_bwd": (C.c_int, [vp, i64, i64, vp, i32, i64, i64, vp, vp, vp, i64, i64, vp, i64, i64, vp, vp, i32, i32, i32,
                                         i32, i32, vp]),
    "b200_causal_conv1d_update": (C.c_int, [vp, i32, i64, i64, i64, vp, i64, i64, i64, vp, i32, i64, i64, vp, i32, i64, vp, i64, i64,
                                            i64, i32, i32, i32, i32, i32, i32, vp]),
    # tests/test_abi.py maps a struct pointer it does not know to c_void_p; the call passes ctypes.byref(SsuParams)
    "b200_selective_state_update": (C.c_int, [vp, vp]),
    "b200_last_error": (C.c_char_p, []),
    "b200_version": (C.c_int, []),
    "b200_kernel_launches": (C.c_int, []),
    "b200_sizeof_params": (C.c_size_t, [i32]),
}
EXPORTS = list(SIGNATURES)

_lib = None


def dtype_code(dt: torch.dtype) -> int:
    try:
        return _DTYPES[dt]
    except KeyError:
        raise RuntimeError(f"libb200ssm: unsupported dtype {dt}") from None


def load() -> C.CDLL:
    """Load (building first if the .so is absent and nvcc is present) -- raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    if _build.can_build():
        _build.build()          # no-op when the digest stamp matches; rebuilds a stale .so after csrc edits (under a file lock)
    elif not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing and nvcc is not available to build it: there is no fallback path")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    for which, st in enumerate((SScanFwdParams, SScanBwdParams, SsdFwdParams, SsdBwdParams, SsuParams)):
        if lib.b200_sizeof_params(which) != C.sizeof(st):
            raise RuntimeError(f"libb200ssm ABI mismatch for {st.__name__}: "
                               f"C {lib.b200_sizeof_params(which)} vs ctypes {C.sizeof(st)}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().b200_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (rc={rc}): {msg}")


def launch(name: str, device, *args) -> None:
    """Call the entry point `name` with `args` and the current stream of `device`, with `device` current; raise on an error."""
    lib = load()
    with torch.cuda.device(device):
        rc = getattr(lib, name)(*args, stream_ptr(device))
    check(rc, name)


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("libb200ssm ops run on CUDA tensors only: there is no CPU fallback")


def f32c(t):
    """t as a detached contiguous fp32 tensor (the layout the kernels read A, D and biases in); None stays None."""
    return None if t is None else t.detach().to(torch.float32).contiguous()


def is_dense(t) -> bool:
    """True when the tensor's elements fill one contiguous block exactly once (any dimension order, e.g. channels_last)."""
    expect = 1
    for size, stride in sorted(((sz, st) for sz, st in zip(t.shape, t.stride()) if sz != 1), key=lambda e: e[1]):
        if stride != expect:
            return False
        expect *= size
    return True


def rows_view(t, D):
    """(tensor, row stride) such that row r of the flattened (..., D) tensor starts at data_ptr + r * stride elements;
    views whose leading dimensions collapse (e.g. one half of a chunk(2, -1)) are used in place."""
    if t.is_contiguous():
        return t, D
    ok = t.dim() >= 2 and t.stride(-1) == 1 and all(t.stride(i) == t.stride(i + 1) * t.shape[i + 1] for i in range(t.dim() - 2))
    return (t, t.stride(-2)) if ok else (t.contiguous(), D)


def no_autocast(fn):
    """Decorator for the forward / backward of every ctypes-backed autograd.Function: the kernels read raw data_ptr()s with a fixed
    dtype, so nothing inside may be re-cast by an enclosing torch.autocast region (loss.backward() called inside the autocast
    block runs the backward under autocast too; a torch.bmm in there would then hand a bf16 buffer to an fp32 kernel)."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        with torch.autocast("cuda", enabled=False):
            return fn(*args, **kwargs)
    return wrapper


def launches() -> int:
    return int(load().b200_kernel_launches())
