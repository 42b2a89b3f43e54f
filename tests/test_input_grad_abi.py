"""sn_psm_backward, sn_hmat_backward and sn_lr_tc_backward reject bad input-gradient arguments with an error code and a message,
before they touch a device (CPU only)."""
import ctypes

from structurednets_b200 import _lib

BUF = ctypes.c_void_p(0x2000)   # never dereferenced: the argument checks fail first


def last_error():
    return _lib.lib().sn_last_error_string()


def psm_factors(in_dim=40, out_dim=24, with_grads=True):
    """One factor (out_dim x in_dim) whose descriptor passes the chain checks; nnz = 0, so no value or column arrays are needed."""
    arr = (_lib.SnPsmFactor * 1)()
    f = arr[0]
    f.rows, f.cols, f.nnz = out_dim, in_dim, 0
    for e, n in ((f.fwd, out_dim), (f.tr, in_dim)):
        e.nslices, e.total = (n + 31) // 32, 0
        e.rowmap = e.slice_off = 0x1000
    f.vals = f.val_fwd = f.val_tr = 0x1000
    if with_grads:
        f.grad_vals = f.grad_packed = 0x1000
    return arr


def psm_backward(arr, grad_x, ldgx, in_dim=40, out_dim=24):
    return _lib.lib().sn_psm_backward(arr, 1, BUF, in_dim, BUF, out_dim, None, None, grad_x, ldgx, 8, in_dim, out_dim, None)


def test_psm_grad_x_with_a_too_small_leading_dimension_is_rejected(built_lib):
    assert psm_backward(psm_factors(), BUF, 39) != 0
    assert b"grad_x leading dimension" in last_error()
    assert psm_backward(psm_factors(with_grads=False), BUF, 3) != 0
    assert b"grad_x leading dimension" in last_error()


def test_psm_no_factor_gradients_and_no_grad_x_is_rejected(built_lib):
    assert psm_backward(psm_factors(with_grads=False), None, 0) != 0
    assert b"both NULL" in last_error()


def test_psm_factor_gradient_buffers_are_all_set_or_all_null(built_lib):
    arr = psm_factors(with_grads=False)
    arr[0].fwd.total, arr[0].fwd.col, arr[0].fwd.src = 32, 0x1000, 0x1000
    arr[0].tr.total, arr[0].tr.col, arr[0].tr.src = 32, 0x1000, 0x1000
    arr[0].grad_vals = 0x1000          # grad_packed missing
    assert psm_backward(arr, BUF, 40) != 0
    assert b"no gradient buffer" in last_error()


def hmat_backward(grad_params, grad_x, ldgx, in_dim=64, out_dim=40):
    return _lib.lib().sn_hmat_backward(BUF, 1, BUF, BUF, in_dim, BUF, out_dim, grad_params, None, grad_x, ldgx, 8, in_dim, out_dim, None)


def test_hmat_grad_x_with_a_too_small_leading_dimension_is_rejected(built_lib):
    assert hmat_backward(BUF, BUF, 63) != 0
    assert b"grad_x leading dimension" in last_error()
    assert hmat_backward(None, BUF, 0) != 0
    assert b"grad_x leading dimension" in last_error()


def test_hmat_no_parameter_gradients_and_no_grad_x_is_rejected(built_lib):
    assert hmat_backward(None, None, 0) != 0
    assert b"both NULL" in last_error()


def lr_tc_backward(grad_x, ldgx, right_bf16=BUF, right_t=BUF, in_dim=40, out_dim=24, rank=16):
    B = ldt = 8
    return _lib.lib().sn_lr_tc_backward(BUF, in_dim, BUF, out_dim, BUF, out_dim, right_bf16, BUF, BUF, BUF, BUF, BUF, BUF, ldt, right_t,
                                        BUF, BUF, None, grad_x, ldgx, B, in_dim, out_dim, rank, None)


def test_lr_tc_grad_x_with_a_too_small_leading_dimension_is_rejected(built_lib):
    assert lr_tc_backward(BUF, 32) != 0
    assert b"grad_x leading dimension too small" in last_error()


def test_lr_tc_grad_x_leading_dimension_must_be_a_multiple_of_8(built_lib):
    assert lr_tc_backward(BUF, 44) != 0
    assert b"not a multiple of 8" in last_error()


def test_lr_tc_grad_x_needs_r_and_its_transpose_scratch(built_lib):
    assert lr_tc_backward(BUF, 40, right_t=None) != 0
    assert b"right_t" in last_error()
    assert lr_tc_backward(BUF, 40, right_bf16=None) != 0
    assert b"right_bf16" in last_error()


def test_lr_tc_transpose_scratch_is_needed_only_for_the_factor_gradients_it_serves(built_lib):
    B = ldt = 8
    call = lambda gyt, xt, gl, gr: _lib.lib().sn_lr_tc_backward(BUF, 40, BUF, 24, BUF, 24, BUF, BUF, BUF, gyt, BUF, BUF, xt, ldt, BUF, gl, gr, None,
                                                                  BUF, 40, B, 40, 24, 16, None)
    assert call(None, BUF, BUF, None) != 0 and b"transpose scratch" in last_error()
    assert call(BUF, None, None, BUF) != 0 and b"transpose scratch" in last_error()
    assert call(None, None, None, BUF) != 0 and b"transpose scratch" in last_error()
