"""bf16 features on the layers that multiply their weight out into a dense matrix (PSM dense-product path, H-matrix dense-block
path, LDR, TL), see csrc/dense_bf16.cu.

W is rebuilt in float32 from the current parameters on every forward by the layer's own kernels; its bf16 copy (and, when the
backward has to return ``grad_x``, its bf16 transpose) is made from that, so nothing bf16 outlives a call.  The batch GEMMs run on
bf16 tensor cores with fp32 accumulation; y and grad_x are bfloat16, parameter gradients float32 as on the float32 path.
Stated tolerance (tests/test_dense_bf16_gpu.py): 2e-2 relative to the largest entry, against the float32 oracle evaluated on the
bf16-rounded features and output gradients.

TMA needs 16-byte aligned operands with a row pitch that is a multiple of 8 bf16: features and output gradients that are not laid
out that way are copied into a padded buffer, outputs are written into one and returned as a view of its first columns.
"""
import torch

from structurednets_b200 import _lib


def pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def _tma_ready(t: torch.Tensor) -> bool:
    return t.stride(1) == 1 and t.stride(0) % 8 == 0 and t.data_ptr() % 16 == 0


def staged(t: torch.Tensor) -> torch.Tensor:
    """``t`` (B x n, bfloat16) itself when the GEMMs can read it, else a copy with a padded row pitch."""
    t = t.to(torch.bfloat16)
    if t.shape[0] == 0 or _tma_ready(t):
        return t
    buf = torch.empty((t.shape[0], pad8(t.shape[1])), dtype=torch.bfloat16, device=t.device)
    buf[:, :t.shape[1]] = t
    return buf[:, :t.shape[1]]


def empty_rows(B: int, n: int, device) -> torch.Tensor:
    """(B x n) bfloat16 output with a row pitch the GEMM epilogue's vector stores and TMA accept."""
    return torch.empty((B, pad8(n)), dtype=torch.bfloat16, device=device)[:, :n]


def weight_buffer(layer, n_out: int, n_in: int, device) -> torch.Tensor:
    """The layer's bf16 W [n_out][pad8(n_in)], cached by device and shape; only read inside the forward that fills it."""
    t = layer.__dict__.get("_dev_W_bf16")
    if t is None or t.device != device or t.shape != (n_out, pad8(n_in)):
        t = torch.empty((n_out, pad8(n_in)), dtype=torch.bfloat16, device=device)
        layer.__dict__["_dev_W_bf16"] = t
    return t


def cast(M: torch.Tensor, Mb, Mtb):
    """Mb = bf16(M) and / or Mtb = bf16(M)^T (either None) in one pass over the float32 M."""
    rows, cols = M.shape
    rc = _lib.lib().sn_dense_cast_bf16(_lib.ptr(M), rows, cols, _lib.ptr(Mb), Mb.stride(0) if Mb is not None else 0, _lib.ptr(Mtb),
                                       Mtb.stride(0) if Mtb is not None else 0, _lib.stream_ptr())
    _lib.check(rc, "sn_dense_cast_bf16")


def forward(layer, W: torch.Tensor, x: torch.Tensor, bias, keep_wt: bool):
    """y = x W^T + bias for the float32 W [n_out][n_in] just built; returns (y, the bf16 W^T for grad_x or None)."""
    n_out, n_in = W.shape
    Wb = weight_buffer(layer, n_out, n_in, x.device)
    Wtb = torch.empty((n_in, pad8(n_out)), dtype=torch.bfloat16, device=x.device) if keep_wt else None
    cast(W, Wb, Wtb)
    return apply(Wb, n_out, x, bias), Wtb


def apply(Wb: torch.Tensor, n_out: int, x: torch.Tensor, bias) -> torch.Tensor:
    B, n_in = x.shape
    y = empty_rows(B, n_out, x.device)
    rc = _lib.lib().sn_dense_apply_bf16(_lib.ptr(Wb), Wb.stride(0), n_out, n_in, _lib.ptr(x), x.stride(0), _lib.ptr(y), y.stride(0), _lib.ptr(bias),
                                        B, _lib.stream_ptr())
    _lib.check(rc, "sn_dense_apply_bf16")
    return y


def weight_grad(x: torch.Tensor, gy: torch.Tensor, dW: torch.Tensor, grad_bias):
    """dW += gy^T x (float32 dW [n_out][n_in]), grad_bias += column sums of gy."""
    n_out, n_in = dW.shape
    rc = _lib.lib().sn_dense_weight_grad_bf16(_lib.ptr(x), x.stride(0), _lib.ptr(gy), gy.stride(0), _lib.ptr(dW), dW.stride(0), n_out, n_in,
                                              _lib.ptr(grad_bias), x.shape[0], _lib.stream_ptr())
    _lib.check(rc, "sn_dense_weight_grad_bf16")


def input_grad(Wtb: torch.Tensor, gy: torch.Tensor) -> torch.Tensor:
    """grad_x = gy W from the bf16 W^T [n_in][ld] kept by the forward."""
    B, n_out = gy.shape
    n_in = Wtb.shape[0]
    gx = empty_rows(B, n_in, gy.device)
    rc = _lib.lib().sn_dense_input_grad_bf16(_lib.ptr(Wtb), Wtb.stride(0), n_out, n_in, _lib.ptr(gy), gy.stride(0), _lib.ptr(gx), gx.stride(0),
                                             B, _lib.stream_ptr())
    _lib.check(rc, "sn_dense_input_grad_bf16")
    return gx
