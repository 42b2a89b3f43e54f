"""ctypes binding of libsnb200.so (the C ABI declared in include/snb200.h).

The product path has no CPU fallback: if the shared library is missing or a kernel reports an
error, a RuntimeError is raised.
"""
import ctypes
import os
from ctypes import c_char_p, c_int, c_int32, c_int64, c_longlong, c_size_t, c_void_p, POINTER, Structure

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libsnb200.so")


class SnSssStage(Structure):
    _fields_ = [(n, c_int32) for n in ("in_off", "in_dim", "out_off", "out_dim", "d_in", "d_out",
                                      "off_ys", "off_yu", "off_ss", "off_su", "pack_off", "k")] + [("reserved", c_int32 * 4)]


class SnSssChunk(Structure):
    _fields_ = [(n, c_int32) for n in ("kk_begin", "kk_end", "col0", "ncols", "row0", "nrows", "second_visit", "kk_mid",
                                      "col0_a", "ncols_a", "col0_b", "ncols_b")] + [("reserved", c_int32 * 4)]


class SnSssPlan(Structure):
    _fields_ = [(n, c_int32) for n in ("nb_states", "input_dim", "output_dim", "rows_pad", "k_pad", "d_pad", "nchunks",
                                      "chunk_in_max", "chunk_out_max", "chunk_len_max", "nparams", "half_in_max")] + \
               [("stages", c_void_p), ("chunks", c_void_p)]


class SnSssTcChunk(Structure):
    _fields_ = [(n, c_int32) for n in ("k_begin", "k_end", "col0", "ncols", "row0", "nrows", "nkb", "reserved")]


class SnSssTcPlan(Structure):
    _fields_ = [(n, c_int32) for n in ("nb_states", "input_dim", "output_dim", "nchunks", "rows_aligned", "chunk_param_floats")] + \
               [("reserved", c_int32 * 2), ("stages", c_void_p), ("chunks", c_void_p)]


class SnPsmEll(Structure):
    _fields_ = [("nslices", c_int32), ("total", c_int32)] + [(n, c_void_p) for n in ("rowmap", "slice_off", "col", "src")]


class SnPsmFactor(Structure):
    _fields_ = [("rows", c_int32), ("cols", c_int32), ("nnz", c_int32), ("reserved", c_int32), ("fwd", SnPsmEll), ("tr", SnPsmEll)] + \
               [(n, c_void_p) for n in ("vals", "grad_vals", "val_fwd", "val_tr", "grad_packed")]


class SnPsmDenseFactor(Structure):
    _fields_ = [("rows", c_int32), ("cols", c_int32), ("nnz", c_int32), ("reserved", c_int32)] + \
               [(n, c_void_p) for n in ("csr_ptr", "csr_idx", "csr_src", "csc_ptr", "csc_idx", "csc_src", "coo_row", "coo_col", "vals", "grad_vals")]


_lib = None


def _declare(lib):
    lib.sn_version.restype = c_int
    lib.sn_last_error_string.restype = c_char_p
    lib.sn_launch_count.restype = c_longlong
    lib.sn_reset_launch_count.restype = None
    lib.sn_timing_enable.restype = None
    lib.sn_timing_enable.argtypes = [c_int]
    lib.sn_timing_report.restype = c_int
    lib.sn_timing_report.argtypes = [c_char_p, c_int]
    P = POINTER(SnSssPlan)
    lib.sn_sss_packed_floats.restype = c_size_t
    lib.sn_sss_packed_floats.argtypes = [P]
    lib.sn_sss_ckpt_floats.restype = c_size_t
    lib.sn_sss_ckpt_floats.argtypes = [P, c_int64]
    lib.sn_sss_pack.restype = c_int
    lib.sn_sss_pack.argtypes = [P, c_void_p, c_void_p, c_void_p]
    lib.sn_sss_forward.restype = c_int
    lib.sn_sss_forward.argtypes = [P, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p]
    lib.sn_sss_backward.restype = c_int
    lib.sn_sss_backward_workspace_floats.restype = c_size_t
    lib.sn_sss_backward_workspace_floats.argtypes = [P]
    lib.sn_sss_backward.argtypes = [P, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_int64, c_int64, c_void_p]
    i64, i32, vp = c_int64, c_int, c_void_p
    PT = POINTER(SnSssTcPlan)
    for name in ("sn_sss_tc_coef_floats",):
        getattr(lib, name).restype = c_size_t
        getattr(lib, name).argtypes = [PT]
    for name in ("sn_sss_tc_rbuf_floats", "sn_sss_tc_states_floats", "sn_sss_tc_backward_workspace_floats"):
        getattr(lib, name).restype = c_size_t
        getattr(lib, name).argtypes = [PT, i64]
    lib.sn_sss_tc_build.restype = c_int
    lib.sn_sss_tc_build.argtypes = [PT, vp, vp, vp]
    lib.sn_sss_tc_forward.restype = c_int
    lib.sn_sss_tc_forward.argtypes = [PT, vp, vp, i64, vp, i64, vp, vp, vp, i64, vp]
    lib.sn_sss_tc_backward.restype = c_int
    lib.sn_sss_tc_backward.argtypes = [PT, vp, vp, vp, i64, vp, i64, vp, vp, vp, vp, vp, i64, i64, vp]
    lib.sn_lr_forward_f32.restype = c_int
    lib.sn_lr_forward_f32.argtypes = [vp, i64, vp, vp, vp, vp, vp, i64, i64, i32, i32, i32, vp]
    lib.sn_lr_backward_f32.restype = c_int
    lib.sn_lr_backward_f32.argtypes = [vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i32, i32, i32, vp]
    lib.sn_hmat_forward.restype = c_int
    lib.sn_hmat_forward.argtypes = [vp, i32, vp, vp, i64, vp, i64, vp, i64, i32, i32, vp]
    lib.sn_hmat_backward.restype = c_int
    lib.sn_hmat_backward.argtypes = [vp, i32, vp, vp, i64, vp, i64, vp, vp, vp, i64, i64, i32, i32, vp]
    lib.sn_hmat_build_dense.restype = c_int
    lib.sn_hmat_build_dense.argtypes = [vp, i32, i32, vp, i32, vp, vp, i32, i32, vp]
    lib.sn_hmat_project_grad.restype = c_int
    lib.sn_hmat_project_grad.argtypes = [vp, i32, vp, i32, vp, vp, i32, i32, vp, vp]
    PF = POINTER(SnPsmFactor)
    lib.sn_psm_forward.restype = c_int
    lib.sn_psm_forward.argtypes = [PF, i32, vp, i64, vp, i64, vp, vp, i64, i32, i32, vp]
    lib.sn_psm_backward.restype = c_int
    lib.sn_psm_backward.argtypes = [PF, i32, vp, i64, vp, i64, vp, vp, vp, i64, i64, i32, i32, vp]
    lib.sn_psm_acts_floats.restype = c_size_t
    lib.sn_psm_acts_floats.argtypes = [PF, i32, i64]
    PD = POINTER(SnPsmDenseFactor)
    lib.sn_psm_dense_prefix_floats.restype = c_size_t
    lib.sn_psm_dense_prefix_floats.argtypes = [PD, i32, i32]
    lib.sn_psm_dense_backward_floats.restype = c_size_t
    lib.sn_psm_dense_backward_floats.argtypes = [PD, i32, i32]
    lib.sn_psm_dense_forward.restype = c_int
    lib.sn_psm_dense_forward.argtypes = [PD, i32, vp, i64, vp, i64, vp, vp, i64, i32, i32, vp]
    lib.sn_psm_dense_backward.restype = c_int
    lib.sn_psm_dense_backward.argtypes = [PD, i32, vp, i64, vp, i64, vp, vp, vp, i64, i32, i32, vp]
    lib.sn_psm_dense_input_grad.restype = c_int
    lib.sn_psm_dense_input_grad.argtypes = [PD, i32, vp, vp, i64, vp, i64, i64, i32, i32, vp]
    f64 = ctypes.c_double
    lib.sn_ldr_workspace_bytes.restype = c_size_t
    lib.sn_ldr_workspace_bytes.argtypes = [i32, i32, i32]
    lib.sn_ldr_build_weight.restype = c_int
    lib.sn_ldr_build_weight.argtypes = [i32, i32, vp, vp, i32, vp, vp, i32, vp, vp, vp, i32, f64, vp, vp, vp]
    lib.sn_ldr_backward.restype = c_int
    lib.sn_ldr_backward.argtypes = [i32, i32, vp, vp, i32, vp, i32, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.sn_dense_input_grad.restype = c_int
    lib.sn_dense_input_grad.argtypes = [vp, i32, i32, vp, i64, vp, i64, i64, vp]
    lib.sn_dense_apply.restype = c_int
    lib.sn_dense_apply.argtypes = [vp, i32, i32, vp, i64, vp, i64, vp, i64, vp]
    lib.sn_dense_weight_grad.restype = c_int
    lib.sn_dense_weight_grad.argtypes = [vp, i64, vp, i64, vp, i32, i32, vp, i64, vp]
    lib.sn_tl_build_weight.restype = c_int
    lib.sn_tl_build_weight.argtypes = [i32, i32, vp, vp, vp, vp, vp, vp]
    lib.sn_tl_backward.restype = c_int
    lib.sn_tl_backward.argtypes = [i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.sn_dense_cast_bf16.restype = c_int
    lib.sn_dense_cast_bf16.argtypes = [vp, i32, i32, vp, i64, vp, i64, vp]
    lib.sn_dense_apply_bf16.restype = c_int
    lib.sn_dense_apply_bf16.argtypes = [vp, i64, i32, i32, vp, i64, vp, i64, vp, i64, vp]
    lib.sn_dense_weight_grad_bf16.restype = c_int
    lib.sn_dense_weight_grad_bf16.argtypes = [vp, i64, vp, i64, vp, i64, i32, i32, vp, i64, vp]
    lib.sn_dense_input_grad_bf16.restype = c_int
    lib.sn_dense_input_grad_bf16.argtypes = [vp, i64, i32, i32, vp, i64, vp, i64, i64, vp]
    lib.sn_psm_dense_forward_bf16.restype = c_int
    lib.sn_psm_dense_forward_bf16.argtypes = [PD, i32, vp, i64, vp, i64, vp, vp, vp, i64, vp, i64, i64, i32, i32, vp]
    lib.sn_psm_dense_backward_bf16.restype = c_int
    lib.sn_psm_dense_backward_bf16.argtypes = [PD, i32, vp, i64, vp, i64, vp, vp, vp, i64, i32, i32, vp]
    lib.sn_lr_tc_cast_params.restype = c_int
    lib.sn_lr_tc_cast_params.argtypes = [vp, vp, vp, vp, i64, vp, i32, i32, i32, vp]
    lib.sn_lr_tc_forward.restype = c_int
    lib.sn_lr_tc_forward.argtypes = [vp, i64, vp, vp, vp, vp, vp, i64, i64, i32, i32, i32, vp]
    lib.sn_lr_tc_backward.restype = c_int
    lib.sn_lr_tc_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, i64, i64, i32, i32, i32, vp]
    f32 = ctypes.c_float
    lib.sn_ce_loss.restype = c_int
    lib.sn_ce_loss.argtypes = [vp, i64, vp, i64, i32, vp, vp, vp, i64, vp]
    lib.sn_mse_loss.restype = c_int
    lib.sn_mse_loss.argtypes = [vp, i64, vp, i64, i64, i32, vp, vp, vp, i64, vp]
    lib.sn_flat_sgd.restype = c_int
    lib.sn_flat_sgd.argtypes = [vp, vp, i64, f32, f32, vp]
    lib.sn_flat_adam.restype = c_int
    lib.sn_flat_adam.argtypes = [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, vp, i32, vp]
    lib.sn_p2p_region_bytes.restype = ctypes.c_size_t
    lib.sn_p2p_region_bytes.argtypes = [i64, c_int]
    lib.sn_p2p_alloc.restype = c_int
    lib.sn_p2p_alloc.argtypes = [ctypes.POINTER(c_void_p), i64, c_int]
    lib.sn_p2p_free.restype = c_int
    lib.sn_p2p_free.argtypes = [vp]
    lib.sn_p2p_export.restype = c_int
    lib.sn_p2p_export.argtypes = [vp, ctypes.c_char_p]
    lib.sn_p2p_import.restype = c_int
    lib.sn_p2p_import.argtypes = [ctypes.c_char_p, ctypes.POINTER(c_void_p)]
    lib.sn_p2p_close.restype = c_int
    lib.sn_p2p_close.argtypes = [vp]
    lib.sn_allreduce_oneshot_f32.restype = c_int
    lib.sn_allreduce_oneshot_f32.argtypes = [vp, i64, ctypes.POINTER(c_void_p), c_int, c_int, i64, f32, vp]
    for name, fn in _EXTRA_DECLS:
        fn(lib)


_EXTRA_DECLS = []  # filled by the other layer modules' declarations below


def lib():
    """The loaded library; raises if it has not been built (python -m structurednets_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libsnb200.so is missing (%s): build it with `python -m structurednets_b200.build`; "
                "structurednets_b200 has no CPU or PyTorch fallback" % LIB_PATH)
        _lib = ctypes.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().sn_last_error_string()
        raise RuntimeError("libsnb200 %s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def timing_report() -> dict:
    """{kernel name: (launches, total ms)} for the launches recorded since the last report (synchronises the device)."""
    import torch
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib().sn_timing_report(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, cnt, ms = line.split()
        out[name] = (int(cnt), float(ms))
    return out


def launch_count() -> int:
    return int(lib().sn_launch_count())


def reset_launch_count():
    lib().sn_reset_launch_count()
