"""Toeplitz-like layer on B200.  Drop-in for ``structurednets.layers.tl_layer.TLLayer`` (reference
layers/tl_layer.py:20-76): square only; parameters ``bias, G (n x r), H (r x n)`` float32 with
``r = int(int(share*n*n) / (2n))``; W = 1/2 sum_j Krylov(Z_1, G[:,j]) Krylov(Z_-1, flip(H[j,:])).
Weight build, apply and backward run in csrc/ldr_tl.cu (``sn_tl_*``, ``sn_dense_*``).
"""
import pickle

import numpy as np
import torch
import torch.nn as nn

from structurednets_b200 import _lib
from structurednets_b200.layers import dense_bf16 as D
from structurednets_b200.layers.flat_params import FlatParamsMixin
from structurednets_b200.layers.layer_helpers import get_random_glorot_uniform_matrix
from structurednets_b200.layers.lr_layer import svd_low_rank_factors
from structurednets_b200.layers.structured_layer import StructuredLayer


def _tl_build_weight(layer, dev):
    """W (n x n, float32) and the Krylov scratch K1, K2 that sn_tl_backward reuses."""
    n, r = layer.G.shape
    K1 = torch.empty((n, n * r), dtype=torch.float32, device=dev)
    K2 = torch.empty((n * r, n), dtype=torch.float32, device=dev)
    W = torch.empty((n, n), dtype=torch.float32, device=dev)
    rc = _lib.lib().sn_tl_build_weight(n, r, _lib.ptr(layer.G), _lib.ptr(layer.H), _lib.ptr(K1), _lib.ptr(K2), _lib.ptr(W), _lib.stream_ptr())
    _lib.check(rc, "sn_tl_build_weight")
    return W, K1, K2


def _tl_param_grads(layer, dW, K1, K2):
    """dW -> G.grad, H.grad (accumulated into the flat gradient buffer)."""
    n, r = layer.G.shape
    dK1, dK2 = torch.empty_like(K1), torch.empty_like(K2)
    rc = _lib.lib().sn_tl_backward(n, r, _lib.ptr(dW), _lib.ptr(K1), _lib.ptr(K2), _lib.ptr(dK1), _lib.ptr(dK2), _lib.ptr(layer.G.grad),
                                   _lib.ptr(layer.H.grad), _lib.stream_ptr())
    _lib.check(rc, "sn_tl_backward")


class _TLFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, U, anchor, layer):
        n, r = layer.G.shape
        dev = U.device
        W, K1, K2 = _tl_build_weight(layer, dev)
        y = torch.empty((U.shape[0], n), dtype=torch.float32, device=dev)
        rc = _lib.lib().sn_dense_apply(_lib.ptr(W), n, n, _lib.ptr(U), U.stride(0), _lib.ptr(y), y.stride(0),
                                       _lib.ptr(layer.bias if layer.use_bias else None), U.shape[0], _lib.stream_ptr())
        _lib.check(rc, "sn_dense_apply")
        ctx.layer = layer
        ctx.save_for_backward(U, K1, K2, W)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        layer = ctx.layer
        U, K1, K2, W = ctx.saved_tensors
        n, r = layer.G.shape
        dev = U.device
        grad_y = grad_y.contiguous().float()
        grad_x = None
        if ctx.needs_input_grad[0]:
            grad_x = torch.empty_like(U)
            _lib.check(_lib.lib().sn_dense_input_grad(_lib.ptr(W), n, n, _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(grad_x), grad_x.stride(0),
                                                      U.shape[0], _lib.stream_ptr()), "sn_dense_input_grad")
        layer._prepare_grad_accumulation()
        dW = torch.zeros((n, n), dtype=torch.float32, device=dev)
        gb = layer.bias.grad if (layer.use_bias and layer.bias.requires_grad) else None
        rc = _lib.lib().sn_dense_weight_grad(_lib.ptr(U), U.stride(0), _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(dW), n, n, _lib.ptr(gb),
                                             U.shape[0], _lib.stream_ptr())
        _lib.check(rc, "sn_dense_weight_grad")
        _tl_param_grads(layer, dW, K1, K2)
        return grad_x, None, None


class _TLBF16Function(torch.autograd.Function):
    """bfloat16 features: the same float32 W, applied and differentiated on bf16 tensor cores (layers/dense_bf16.py)."""

    @staticmethod
    def forward(ctx, U, anchor, layer):
        W, K1, K2 = _tl_build_weight(layer, U.device)
        x = D.staged(U)
        y, Wtb = D.forward(layer, W, x, layer.bias if layer.use_bias else None, keep_wt=ctx.needs_input_grad[0])
        ctx.layer = layer
        ctx.save_for_backward(x, K1, K2, Wtb)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        layer = ctx.layer
        x, K1, K2, Wtb = ctx.saved_tensors
        n = layer.G.shape[0]
        gy = D.staged(grad_y)
        grad_x = D.input_grad(Wtb, gy) if ctx.needs_input_grad[0] else None
        layer._prepare_grad_accumulation()
        dW = torch.zeros((n, n), dtype=torch.float32, device=x.device)
        D.weight_grad(x, gy, dW, layer.bias.grad if (layer.use_bias and layer.bias.requires_grad) else None)
        _tl_param_grads(layer, dW, K1, K2)
        return grad_x, None, None


class TLLayer(FlatParamsMixin, StructuredLayer):
    def __init__(self, input_dim: int, output_dim: int, nb_params_share: float, use_bias=True, initial_weight_matrix=None,
                 initial_bias=None, initial_lr_matrices=None):
        super(TLLayer, self).__init__(input_dim=input_dim, output_dim=output_dim, nb_params_share=nb_params_share, use_bias=use_bias,
                                      initial_weight_matrix=initial_weight_matrix, initial_bias=initial_bias)
        assert input_dim == output_dim, "The TL Layer is only implemented for square weight matrices (i.e. when the number of inputs equals the number of outputs)"
        assert initial_weight_matrix is None or initial_lr_matrices is None, "Either pass an initial weight matrix or initial low rank matrices - not both"
        if initial_lr_matrices is not None:
            assert len(initial_lr_matrices) == 2, "Expect the length of the list of initial low rank matrices to be 2"

        self.input_dim = input_dim
        self.target_mat_shape = (self.output_dim, input_dim)

        if initial_lr_matrices is not None:
            G = pickle.loads(pickle.dumps(initial_lr_matrices[0]))
            H = pickle.loads(pickle.dumps(initial_lr_matrices[1]))
        elif initial_weight_matrix is not None:
            G, H = tl_displacement_factors(initial_weight_matrix, nb_params_share)
        else:
            max_nb_parameters = int(nb_params_share * input_dim * output_dim)
            displacement_rank = int(max_nb_parameters / (input_dim + output_dim))
            G = get_random_glorot_uniform_matrix((output_dim, displacement_rank))
            H = get_random_glorot_uniform_matrix((displacement_rank, input_dim))

        self.G = nn.Parameter(torch.tensor(np.asarray(G)).float())
        self.H = nn.Parameter(torch.tensor(np.asarray(H)).float())
        self._flatten_parameters()

    def forward(self, U):
        displacement_rank = self.G.shape[1]
        if displacement_rank > 0:
            self._require_cuda(U, "TLLayer.forward")
            assert U.dim() == 2 and U.shape[1] == self.input_dim, "TLLayer expects a (batch, input_dim) input"
            self._ensure_flat()
            if U.dtype == torch.bfloat16:     # bf16 output, float32 parameters and gradients
                fn = _TLBF16Function
            else:
                fn = _TLFunction
                if U.dtype != torch.float32:
                    U = U.float()
                if U.stride(1) != 1:
                    U = U.contiguous()
            anchor = self.__dict__.get("_dev_anchor")
            if anchor is None or anchor.device != U.device:
                anchor = torch.zeros(1, device=U.device, requires_grad=True)
                self.__dict__["_dev_anchor"] = anchor
            return fn.apply(U, anchor if torch.is_grad_enabled() else None, self)
        y_pred = torch.zeros((U.shape[0], self.output_dim), device=U.device)   # reference tl_layer.py:62-63
        if self.use_bias:
            y_pred = y_pred + self.bias
        return y_pred

    def get_nb_parameters(self) -> int:
        res = torch.numel(self.G) + torch.numel(self.H)
        if self.use_bias:
            res += torch.numel(self.bias)
        return int(res)


def tl_displacement_factors(optim_mat: np.ndarray, nb_params_share: float):
    """Analytic Toeplitz-like fit of the reference (approximators/tl_approximator.py:39-61): low-rank factors of
    the Sylvester displacement Z_1 W - W Z_-1."""
    n = optim_mat.shape[0]
    Z1 = np.diag(np.ones(n - 1), k=-1); Z1[0, -1] = 1.0
    Zm = np.diag(np.ones(n - 1), k=-1); Zm[0, -1] = -1.0
    disp = Z1 @ optim_mat - optim_mat @ Zm
    rank = int(int(nb_params_share * disp.size) / (2 * n))
    return svd_low_rank_factors(disp, rank)
