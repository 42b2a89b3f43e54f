"""The bf16 dense-product entries (csrc/dense_bf16.cu, csrc/psm.cu) reject NULL buffers with an error code and a message instead of
faulting or throwing across the C boundary (argument checks run before anything touches a device: CPU only)."""
from structurednets_b200 import _lib


def test_bf16_dense_entries_reject_null_buffers(built_lib):
    lib = _lib.lib()
    calls = {
        "sn_dense_cast_bf16": lambda: lib.sn_dense_cast_bf16(None, 4, 4, None, 8, None, 8, None),
        "sn_dense_apply_bf16": lambda: lib.sn_dense_apply_bf16(None, 8, 4, 4, None, 8, None, 8, None, 4, None),
        "sn_dense_weight_grad_bf16": lambda: lib.sn_dense_weight_grad_bf16(None, 8, None, 8, None, 4, 4, 4, None, 4, None),
        "sn_dense_input_grad_bf16": lambda: lib.sn_dense_input_grad_bf16(None, 8, 4, 4, None, 8, None, 8, 4, None),
        "sn_psm_dense_forward_bf16": lambda: lib.sn_psm_dense_forward_bf16(None, 0, None, 8, None, 8, None, None, None, 8, None, 8, 4, 4, 4, None),
        "sn_psm_dense_backward_bf16": lambda: lib.sn_psm_dense_backward_bf16(None, 0, None, 8, None, 8, None, None, None, 4, 4, 4, None),
    }
    for name, call in calls.items():
        rc = call()
        msg = lib.sn_last_error_string()
        assert rc != 0, name
        assert msg and (b"NULL" in msg or b"psm_dense" in msg), (name, msg)
