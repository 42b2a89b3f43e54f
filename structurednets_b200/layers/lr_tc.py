"""bf16 tensor-core path of the low-rank layer (BASELINE config C2), see csrc/lr_tc.cu / csrc/gemm_tc.cuh.

Selected by ``LRLayer.forward`` when the features are bfloat16.  Parameters stay float32 (master copies in the
layer's flat buffer); bf16 copies are refreshed on every forward (one small launch).  Output and the kept hidden
activations are bfloat16, accumulation is float32 in TMEM, parameter gradients are accumulated in float32.
Stated tolerance (tests/test_lr_tc_gpu.py): 2e-2 relative to the largest entry, against the float32 oracle.
"""
import torch

from structurednets_b200 import _lib
from structurednets_b200.layers import dense_bf16 as D


def _bf16_params(layer):
    flat = layer.flat_parameters()
    cache = layer.__dict__.get("_dev_bf16")
    out_dim, rank = layer.left_lr.shape
    in_dim = layer.right_lr.shape[1]
    if cache is None or cache["device"] != flat.device:
        lt_ld = (out_dim + 7) // 8 * 8
        cache = dict(device=flat.device, version=None, lt_ld=lt_ld,
                     L=torch.empty((out_dim, rank), dtype=torch.bfloat16, device=flat.device),
                     Lt=torch.zeros((rank, lt_ld), dtype=torch.bfloat16, device=flat.device),
                     R=torch.empty((rank, in_dim), dtype=torch.bfloat16, device=flat.device))
        layer.__dict__["_dev_bf16"] = cache
    if True:   # refreshed on every forward: in-place optimizer updates are not otherwise detectable cheaply
        rc = _lib.lib().sn_lr_tc_cast_params(_lib.ptr(layer.left_lr), _lib.ptr(layer.right_lr), _lib.ptr(cache["L"]), _lib.ptr(cache["Lt"]),
                                             cache["lt_ld"], _lib.ptr(cache["R"]), in_dim, out_dim, rank, _lib.stream_ptr())
        _lib.check(rc, "sn_lr_tc_cast_params")
    return cache


class _LRFunctionBF16(torch.autograd.Function):
    @staticmethod
    def forward(ctx, U, anchor, layer):
        B = U.shape[0]
        out_dim, rank = layer.left_lr.shape
        in_dim = layer.right_lr.shape[1]
        P = _bf16_params(layer)
        ldy = (out_dim + 7) // 8 * 8
        hidden = torch.empty((B, rank), dtype=torch.bfloat16, device=U.device)
        ybuf = torch.empty((B, ldy), dtype=torch.bfloat16, device=U.device)
        rc = _lib.lib().sn_lr_tc_forward(_lib.ptr(U), U.stride(0), _lib.ptr(P["L"]), _lib.ptr(P["R"]), _lib.ptr(layer.bias if layer.use_bias else None),
                                         _lib.ptr(hidden), _lib.ptr(ybuf), ldy, B, in_dim, out_dim, rank, _lib.stream_ptr())
        _lib.check(rc, "sn_lr_tc_forward")
        ctx.layer = layer
        ctx.P = P
        ctx.save_for_backward(U, hidden)
        return ybuf[:, :out_dim]

    @staticmethod
    def backward(ctx, grad_y):
        layer = ctx.layer
        U, hidden = ctx.saved_tensors
        B = U.shape[0]
        out_dim, rank = layer.left_lr.shape
        in_dim = layer.right_lr.shape[1]
        P = ctx.P
        gy = grad_y.to(torch.bfloat16)
        if gy.stride(1) != 1 or gy.stride(0) % 8 != 0 or gy.data_ptr() % 16 != 0:
            ldg = (out_dim + 7) // 8 * 8
            buf = torch.empty((B, ldg), dtype=torch.bfloat16, device=U.device)
            buf[:, :out_dim] = gy
            gy = buf[:, :out_dim]
        if any(p.requires_grad for p in layer._flat_param_list()):   # a frozen layer never allocates the flat gradient buffer
            layer._prepare_grad_accumulation()
        ldt = (B + 7) // 8 * 8
        mk = lambda rows: torch.empty((rows, ldt), dtype=torch.bfloat16, device=U.device)
        ghid = torch.empty((B, rank), dtype=torch.bfloat16, device=U.device)
        gl = layer.left_lr.grad if layer.left_lr.requires_grad else None
        gr = layer.right_lr.grad if layer.right_lr.requires_grad else None
        # transpose scratch of the dL / dR GEMMs, only for the factors that take a gradient
        gyt, ht = (mk(out_dim), mk(rank)) if gl is not None else (None, None)
        ght, xt = (mk(rank), mk(in_dim)) if gr is not None else (None, None)
        gb = layer.bias.grad if (layer.use_bias and layer.bias.requires_grad) else None
        grad_x = rt = None
        if ctx.needs_input_grad[0]:   # grad_x = ghid R, bf16 like the features (rows padded to 16 bytes for the GEMM's stores)
            grad_x = D.empty_rows(B, in_dim, U.device)
            rt = torch.empty((in_dim, rank), dtype=torch.bfloat16, device=U.device)
        rc = _lib.lib().sn_lr_tc_backward(_lib.ptr(U), U.stride(0), _lib.ptr(gy), gy.stride(0), _lib.ptr(P["Lt"]), P["lt_ld"], _lib.ptr(P["R"]),
                                          _lib.ptr(hidden), _lib.ptr(ghid), _lib.ptr(gyt), _lib.ptr(ht), _lib.ptr(ght), _lib.ptr(xt), ldt, _lib.ptr(rt),
                                          _lib.ptr(gl), _lib.ptr(gr), _lib.ptr(gb), _lib.ptr(grad_x), grad_x.stride(0) if grad_x is not None else 0,
                                          B, in_dim, out_dim, rank, _lib.stream_ptr())
        _lib.check(rc, "sn_lr_tc_backward")
        return grad_x, None, None


def lr_forward_bf16(layer, U, anchor):
    rank = layer.left_lr.shape[1]
    if rank % 8 != 0 or rank < 8:
        raise RuntimeError("LRLayer (bf16 tensor-core path) needs rank %% 8 == 0, got rank %d; use float32 features" % rank)
    if U.stride(0) % 8 != 0 or U.data_ptr() % 16 != 0:
        raise RuntimeError("LRLayer (bf16 tensor-core path) needs 16-byte aligned feature rows (row pitch multiple of 8 bf16)")
    return _LRFunctionBF16.apply(U, anchor, layer)
