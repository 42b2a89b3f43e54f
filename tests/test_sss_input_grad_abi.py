"""sn_sss_backward rejects bad input-gradient arguments with an error code and a message, before it touches a device (CPU only)."""
import ctypes

from structurednets_b200 import _lib


def fake_plan(input_dim=40, output_dim=12):
    """A plan that passes the entry's plan checks; its table pointers are never dereferenced because the call fails first."""
    p = _lib.SnSssPlan()
    p.nb_states, p.input_dim, p.output_dim = 4, input_dim, output_dim
    p.rows_pad, p.k_pad, p.d_pad = 8, 16, 4
    p.nchunks, p.chunk_in_max, p.chunk_out_max, p.chunk_len_max = 2, 20, 6, 2
    p.nparams, p.half_in_max = 100, 10
    p.stages = p.chunks = 0x1000
    return p


def backward(plan, grad_params, workspace, grad_x, ldgx):
    buf = ctypes.c_void_p(0x2000)   # never dereferenced: the argument checks fail first
    return _lib.lib().sn_sss_backward(ctypes.byref(plan), buf, buf, plan.input_dim, buf, plan.output_dim, buf, workspace, grad_params,
                                      None, grad_x, ldgx, 8, None)


def test_grad_x_with_a_too_small_leading_dimension_is_rejected(built_lib):
    plan = fake_plan()
    buf = ctypes.c_void_p(0x2000)
    assert backward(plan, buf, buf, buf, plan.input_dim - 1) != 0
    assert b"grad_x leading dimension" in _lib.lib().sn_last_error_string()
    assert backward(plan, None, None, buf, 3) != 0
    assert b"grad_x leading dimension" in _lib.lib().sn_last_error_string()


def test_no_parameter_gradients_and_no_grad_x_is_rejected(built_lib):
    plan = fake_plan()
    assert backward(plan, None, None, None, 0) != 0
    assert b"both NULL" in _lib.lib().sn_last_error_string()
    assert backward(plan, None, ctypes.c_void_p(0x2000), None, plan.input_dim) != 0
    assert b"both NULL" in _lib.lib().sn_last_error_string()


def test_parameter_gradients_need_a_workspace(built_lib):
    plan = fake_plan()
    buf = ctypes.c_void_p(0x2000)
    assert backward(plan, buf, None, buf, plan.input_dim) != 0
    assert b"workspace" in _lib.lib().sn_last_error_string()
