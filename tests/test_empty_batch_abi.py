"""Every batch entry of the C ABI treats an empty batch (B = 0) as a no-op that returns 0 (CPU only).

An empty torch tensor has data_ptr() == 0, and an empty slice of a real tensor has a pointer that must not be read, so each entry is
called twice: with NULL batch buffers and with dummy non-NULL ones that point into the never-mapped first page.  Parameters, plans
and the parameter-gradient buffers get dummy pointers too; their checks run before the batch test and must still pass.  Nothing may
be dereferenced on the host and no CUDA call may be made, so this runs without a GPU.

Each call runs in a subprocess: an entry that crashes (an integer division by zero on the host, a read through a dummy pointer)
shows up as one failing case with its signal instead of ending the test session.
"""
import ctypes
import os
import signal
import subprocess
import sys

import pytest

from structurednets_b200 import _lib

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAM = 0x1000      # parameters, plans' tables, parameter gradients: checked for NULL before B, never dereferenced here
DUMMY = 0x100       # non-NULL batch buffer in the unmapped first page: a host read of it crashes
N_IN, N_OUT, RANK = 40, 24, 16


def _psm_factors():
    arr = (_lib.SnPsmFactor * 1)()
    f = arr[0]
    f.rows, f.cols, f.nnz = N_OUT, N_IN, 0
    for e, n in ((f.fwd, N_OUT), (f.tr, N_IN)):
        e.nslices, e.total = (n + 31) // 32, 0
        e.rowmap = e.slice_off = PARAM
    f.vals = f.val_fwd = f.val_tr = f.grad_vals = f.grad_packed = PARAM
    return arr


def _psm_dense_factors():
    arr = (_lib.SnPsmDenseFactor * 1)()
    f = arr[0]
    f.rows, f.cols, f.nnz = N_OUT, N_IN, 0
    for name in ("csr_ptr", "csr_idx", "csr_src", "csc_ptr", "csc_idx", "csc_src", "coo_row", "coo_col", "vals", "grad_vals"):
        setattr(f, name, PARAM)
    return arr


def _sss_plan():
    p = _lib.SnSssPlan()
    p.nb_states, p.input_dim, p.output_dim = 4, N_IN, N_OUT
    p.rows_pad, p.k_pad, p.d_pad, p.nchunks = 8, 16, 4, 1
    p.chunk_in_max, p.chunk_out_max, p.chunk_len_max, p.nparams, p.half_in_max = N_IN, N_OUT, 4, 64, N_IN
    p.stages = p.chunks = PARAM
    return ctypes.byref(p), p


def _sss_tc_plan():
    p = _lib.SnSssTcPlan()
    p.nb_states, p.input_dim, p.output_dim, p.nchunks = 4, N_IN, N_OUT, 1
    p.rows_aligned, p.chunk_param_floats = 1, 64
    p.stages = p.chunks = PARAM
    return ctypes.byref(p), p


# name -> call(b): b = the pointer every batch buffer gets (None or DUMMY); every call has B = 0
ENTRIES = {
    "sn_dense_apply": lambda L, b: L.sn_dense_apply(PARAM, N_OUT, N_IN, b, N_IN, b, N_OUT, PARAM, 0, None),
    "sn_dense_input_grad": lambda L, b: L.sn_dense_input_grad(PARAM, N_OUT, N_IN, b, N_OUT, b, N_IN, 0, None),
    "sn_dense_weight_grad": lambda L, b: L.sn_dense_weight_grad(b, N_IN, b, N_OUT, PARAM, N_OUT, N_IN, PARAM, 0, None),
    "sn_dense_apply_bf16": lambda L, b: L.sn_dense_apply_bf16(PARAM, N_IN, N_OUT, N_IN, b, N_IN, b, N_OUT, PARAM, 0, None),
    "sn_dense_weight_grad_bf16": lambda L, b: L.sn_dense_weight_grad_bf16(b, N_IN, b, N_OUT, PARAM, N_IN, N_OUT, N_IN, PARAM, 0, None),
    "sn_dense_input_grad_bf16": lambda L, b: L.sn_dense_input_grad_bf16(PARAM, N_OUT, N_OUT, N_IN, b, N_OUT, b, N_IN, 0, None),
    "sn_lr_forward_f32": lambda L, b: L.sn_lr_forward_f32(b, N_IN, PARAM, PARAM, PARAM, b, b, N_OUT, 0, N_IN, N_OUT, RANK, None),
    "sn_lr_backward_f32": lambda L, b: L.sn_lr_backward_f32(b, N_IN, b, N_OUT, PARAM, PARAM, b, b, PARAM, PARAM, PARAM, b, N_IN, 0,
                                                            N_IN, N_OUT, RANK, None),
    "sn_lr_tc_forward": lambda L, b: L.sn_lr_tc_forward(b, N_IN, PARAM, PARAM, PARAM, b, b, N_OUT, 0, N_IN, N_OUT, RANK, None),
    "sn_lr_tc_backward": lambda L, b: L.sn_lr_tc_backward(b, N_IN, b, N_OUT, PARAM, N_OUT, PARAM, b, b, b, b, b, b, 0, PARAM,
                                                          PARAM, PARAM, PARAM, b, N_IN, 0, N_IN, N_OUT, RANK, None),
    "sn_hmat_forward": lambda L, b: L.sn_hmat_forward(PARAM, 1, PARAM, b, N_IN, b, N_OUT, PARAM, 0, N_IN, N_OUT, None),
    "sn_hmat_backward": lambda L, b: L.sn_hmat_backward(PARAM, 1, PARAM, b, N_IN, b, N_OUT, PARAM, PARAM, b, N_IN, 0, N_IN, N_OUT, None),
    "sn_psm_forward": lambda L, b: L.sn_psm_forward(_psm_factors(), 1, b, N_IN, b, N_OUT, PARAM, b, 0, N_IN, N_OUT, None),
    "sn_psm_backward": lambda L, b: L.sn_psm_backward(_psm_factors(), 1, b, N_IN, b, N_OUT, b, PARAM, b, N_IN, 0, N_IN, N_OUT, None),
    "sn_psm_dense_forward": lambda L, b: L.sn_psm_dense_forward(_psm_dense_factors(), 1, b, N_IN, b, N_OUT, PARAM, PARAM, 0, N_IN, N_OUT,
                                                                None),
    "sn_psm_dense_input_grad": lambda L, b: L.sn_psm_dense_input_grad(_psm_dense_factors(), 1, PARAM, b, N_OUT, b, N_IN, 0, N_IN, N_OUT,
                                                                      None),
    "sn_psm_dense_backward": lambda L, b: L.sn_psm_dense_backward(_psm_dense_factors(), 1, b, N_IN, b, N_OUT, PARAM, PARAM, PARAM, 0, N_IN,
                                                                  N_OUT, None),
    "sn_psm_dense_forward_bf16": lambda L, b: L.sn_psm_dense_forward_bf16(_psm_dense_factors(), 1, b, N_IN, b, N_OUT, PARAM, PARAM, PARAM,
                                                                          N_IN, PARAM, N_OUT, 0, N_IN, N_OUT, None),
    "sn_psm_dense_backward_bf16": lambda L, b: L.sn_psm_dense_backward_bf16(_psm_dense_factors(), 1, b, N_IN, b, N_OUT, PARAM, PARAM, PARAM,
                                                                            0, N_IN, N_OUT, None),
    "sn_sss_forward": lambda L, b: L.sn_sss_forward(_sss_plan()[0], PARAM, b, N_IN, b, N_OUT, PARAM, b, 0, None),
    "sn_sss_backward": lambda L, b: L.sn_sss_backward(_sss_plan()[0], PARAM, b, N_IN, b, N_OUT, b, PARAM, PARAM, PARAM, b, N_IN, 0, None),
    "sn_sss_tc_forward": lambda L, b: L.sn_sss_tc_forward(_sss_tc_plan()[0], PARAM, b, N_IN, b, N_OUT, PARAM, b, b, 0, None),
    "sn_sss_tc_backward": lambda L, b: L.sn_sss_tc_backward(_sss_tc_plan()[0], PARAM, PARAM, b, N_IN, b, N_OUT, b, b, PARAM, PARAM, b,
                                                            N_IN, 0, None),
}


def _run(name: str, mode: str) -> None:
    """Subprocess body: one call, then its return code and error message on stdout."""
    lib = _lib.lib()
    rc = ENTRIES[name](lib, None if mode == "null" else DUMMY)
    msg = lib.sn_last_error_string() if rc else b""
    print("rc=%d %s" % (rc, msg.decode(errors="replace")), flush=True)


@pytest.mark.parametrize("mode", ["null", "dummy"])
@pytest.mark.parametrize("name", sorted(ENTRIES))
def test_empty_batch_is_a_no_op(built_lib, name, mode):
    code = "import sys; sys.path.insert(0, %r); from tests import test_empty_batch_abi as t; t._run(%r, %r)" % (REPO, name, mode)
    proc = subprocess.run([sys.executable, "-c", code], cwd=REPO, capture_output=True, text=True, timeout=120)
    if proc.returncode < 0:
        pytest.fail("%s(B = 0, %s batch buffers) died with %s\n%s" % (name, mode, signal.Signals(-proc.returncode).name, proc.stderr[-2000:]))
    assert proc.returncode == 0, proc.stderr[-2000:]
    assert proc.stdout.strip() == "rc=0", "%s(B = 0, %s batch buffers) returned %s" % (name, mode, proc.stdout.strip())
