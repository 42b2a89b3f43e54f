"""Low-displacement-rank layer on B200.  Drop-in for ``structurednets.layers.ldr_layer.LDRLayer``
(reference layers/ldr_layer.py:11-71 and approximators/ldr_approximator.py:8-47): square only
(``assert input_dim == output_dim``), parameters ``bias`` (float32) and ``representation_matrices.{0..3}`` =
A, B (float64 sparse COO, tridiagonal plus two corners, 3n entries) and G, H (float64, n x r); the rank
formula and the "displacement rank < 0 -> dummy parameter, zero output" rule are kept.

The weight is built by csrc/ldr_tl.cu: float64 Krylov recurrences (O(n r) per power) and one tensor-core contraction
over the powers that matter -- the same matrix as the reference's matrix_power construction (O(r n^4 log n)) -- and
applied with fp32-accurate tensor-core GEMMs.
"""
import pickle

import numpy as np
import torch
import torch.nn as nn

from structurednets_b200 import _lib
from structurednets_b200.layers import dense_bf16 as D
from structurednets_b200.layers.layer_helpers import get_random_glorot_uniform_matrix_torch
from structurednets_b200.layers.structured_layer import StructuredLayer

LDR_REL_TOL = 1e-14          # a Krylov power whose bound is this small relative to the largest one cannot change the float32 weight
LDR_TERMS_START = 32         # powers computed by default; quadrupled (up to n) whenever the device reports "not converged"


def get_max_ld_rank_wrt_max_nb_free_parameters(max_nb_free_parameters: int, target_shape_mat: tuple):
    """reference approximators/ldr_approximator.py:8-10"""
    n = min(target_shape_mat)
    return int((max_nb_free_parameters - 2 * (3 * n - 2) + 4) / (2 * n))


def get_nb_free_parameters(displacement_rank: int, target_mat_shape: tuple):
    """reference approximators/ldr_approximator.py:12-14"""
    n = min(target_mat_shape)
    return displacement_rank * 2 * n + 2 * (3 * n - 2) + 4


def get_init_tridiagonal_matrix_with_corners_torch(shape: tuple):
    """reference approximators/ldr_approximator.py:16-27: COO entry order = super-diagonal, sub-diagonal,
    diagonal, the two corners; values U(-limit, limit) with limit sqrt(6/(n+n)), float64."""
    assert shape[0] == shape[1], "get_init_tridiagonal_matrix is only defined for square matrix shapes"
    n = shape[0]
    i = np.arange(n)
    rows = np.concatenate([i[1:] - 1, i[:-1] + 1, i, [0, n - 1]])
    cols = np.concatenate([i[1:], i[:-1], i, [n - 1, 0]])
    limit = np.sqrt(6.0 / (shape[0] + shape[1]))
    vals = np.random.uniform(-limit, limit, size=(3 * n,))
    mat = torch.sparse_coo_tensor(torch.tensor(np.stack([rows, cols])), torch.tensor(vals), shape)
    mat.requires_grad_()
    return mat


def init_representation_matrices_torch(shape: tuple, displacement_rank: int):
    """reference approximators/ldr_approximator.py:41-47"""
    return [get_init_tridiagonal_matrix_with_corners_torch(shape), get_init_tridiagonal_matrix_with_corners_torch(shape),
            get_random_glorot_uniform_matrix_torch((shape[0], displacement_rank)),
            get_random_glorot_uniform_matrix_torch((shape[0], displacement_rank))]


def band_slots(indices: torch.Tensor, n: int) -> torch.Tensor:
    """COO entry -> slot of the banded layout of csrc/ldr_tl.cu (lo | di | up | corner(0,n-1), corner(n-1,0))."""
    r, c = indices[0].long(), indices[1].long()
    slot = torch.full_like(r, -1)
    slot = torch.where(c == r, n + r, slot)
    slot = torch.where(c == r + 1, 2 * n + r, slot)
    slot = torch.where(c == r - 1, r, slot)
    if n > 2:
        slot = torch.where((r == 0) & (c == n - 1), torch.full_like(r, 3 * n), slot)
        slot = torch.where((r == n - 1) & (c == 0), torch.full_like(r, 3 * n + 1), slot)
    if bool((slot < 0).any()):
        raise ValueError("LDRLayer: A and B must be tridiagonal plus the (0,n-1)/(n-1,0) corners "
                         "(approximators/ldr_approximator.py:16-27); found an entry outside that pattern")
    return slot.to(torch.int32).contiguous()


def _ldr_build_weight(layer, dev, A, Bm, G, H):
    """W (n x n, float32) from the representation, with the workspace, status word and term count the backward needs.  Nothing here
    synchronises while a CUDA graph is being captured; outside a capture the 16-byte status word is read back after the Krylov
    kernels so that a series longer than the powers computed is re-run with more (and ``last_nb_terms`` stays observable)."""
    n, r = G.shape
    L = _lib.lib()
    slots = layer._slots(A, Bm)
    Av, Bv = A._values().contiguous(), Bm._values().contiguous()
    Gc, Hc = G.contiguous(), H.contiguous()
    assert Av.dtype == torch.float64 and Gc.dtype == torch.float64, "LDR representation matrices are float64 (SURVEY.md F4)"
    W = torch.empty((n, n), dtype=torch.float32, device=dev)
    status = torch.zeros(4, dtype=torch.int32, device=dev)
    capturing = torch.cuda.is_current_stream_capturing()
    max_terms = min(n, 1024, int(layer.__dict__.get("_terms_cap", LDR_TERMS_START)))
    while True:
        ws = torch.empty(int(L.sn_ldr_workspace_bytes(n, r, max_terms)), dtype=torch.uint8, device=dev)
        rc = L.sn_ldr_build_weight(n, r, _lib.ptr(Av), _lib.ptr(slots[0]), Av.numel(), _lib.ptr(Bv), _lib.ptr(slots[1]), Bv.numel(),
                                   _lib.ptr(Gc), _lib.ptr(Hc), _lib.ptr(ws), max_terms, LDR_REL_TOL, _lib.ptr(W), _lib.ptr(status), _lib.stream_ptr())
        _lib.check(rc, "sn_ldr_build_weight")
        if capturing:
            break
        st = status.tolist()
        layer.last_nb_terms = int(st[0])
        if st[2] or max_terms >= min(n, 1024):
            if st[2]:   # next call computes a few powers more than this one needed, not LDR_TERMS_START
                layer.__dict__["_terms_cap"] = min(n, 1024, max(8, (int(st[0]) + 4 + 3) // 4 * 4))
            if not st[2]:
                raise RuntimeError("LDRLayer: the Krylov series of this (A, B) has not decayed after %d powers (n = %d); the operators' "
                                   "norms are too close to (or above) 1 for the truncated construction" % (max_terms, n))
            break
        max_terms = min(n, 1024, max_terms * 4)
        layer.__dict__["_terms_cap"] = max_terms
    return W, ws, status, max_terms, slots, Gc, Hc


def _ldr_param_grads(dW, slots, ws, max_terms, status, A, Bm, G, H):
    """dW -> sparse dA, dB on the parameters' own pattern (SURVEY.md F4) and dense dG, dH, all float64."""
    n, r = G.shape
    dev = dW.device
    gA = torch.zeros(A._nnz(), dtype=torch.float64, device=dev)
    gB = torch.zeros(Bm._nnz(), dtype=torch.float64, device=dev)
    gG, gH = torch.zeros_like(G), torch.zeros_like(H)
    rc = _lib.lib().sn_ldr_backward(n, r, _lib.ptr(dW), _lib.ptr(slots[0]), gA.numel(), _lib.ptr(slots[1]), gB.numel(), _lib.ptr(ws),
                                    max_terms, _lib.ptr(status), _lib.ptr(gA), _lib.ptr(gB), _lib.ptr(gG), _lib.ptr(gH), _lib.stream_ptr())
    _lib.check(rc, "sn_ldr_backward")
    return torch.sparse_coo_tensor(A._indices(), gA, A.shape), torch.sparse_coo_tensor(Bm._indices(), gB, Bm.shape), gG, gH


class _LDRFunction(torch.autograd.Function):
    """sn_ldr_build_weight + sn_dense_apply / sn_dense_weight_grad + sn_ldr_backward (csrc/ldr_tl.cu), see _ldr_build_weight."""

    @staticmethod
    def forward(ctx, U, bias, layer, A, Bm, G, H):
        n, r = G.shape
        dev = U.device
        L = _lib.lib()
        W, ws, status, max_terms, slots, Gc, Hc = _ldr_build_weight(layer, dev, A, Bm, G, H)
        y = torch.empty((U.shape[0], n), dtype=torch.float32, device=dev)
        rc = L.sn_dense_apply(_lib.ptr(W), n, n, _lib.ptr(U), U.stride(0), _lib.ptr(y), y.stride(0), _lib.ptr(bias), U.shape[0], _lib.stream_ptr())
        _lib.check(rc, "sn_dense_apply")
        ctx.max_terms, ctx.slots, ctx.has_bias = max_terms, slots, bias is not None
        ctx.save_for_backward(U, ws, status, W, A, Bm, Gc, Hc)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        U, ws, status, W, A, Bm, G, H = ctx.saved_tensors
        n, r = G.shape
        dev = U.device
        L = _lib.lib()
        grad_y = grad_y.contiguous().float()
        grad_x = None
        if ctx.needs_input_grad[0]:
            grad_x = torch.empty_like(U)
            _lib.check(L.sn_dense_input_grad(_lib.ptr(W), n, n, _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(grad_x), grad_x.stride(0),
                                             U.shape[0], _lib.stream_ptr()), "sn_dense_input_grad")
        dW = torch.zeros((n, n), dtype=torch.float32, device=dev)
        gbias = torch.zeros(n, dtype=torch.float32, device=dev) if ctx.has_bias else None
        rc = L.sn_dense_weight_grad(_lib.ptr(U), U.stride(0), _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(dW), n, n, _lib.ptr(gbias),
                                    U.shape[0], _lib.stream_ptr())
        _lib.check(rc, "sn_dense_weight_grad")
        gAs, gBs, gG, gH = _ldr_param_grads(dW, ctx.slots, ws, ctx.max_terms, status, A, Bm, G, H)
        return grad_x, gbias, None, gAs, gBs, gG, gH


class _LDRBF16Function(torch.autograd.Function):
    """bfloat16 features: the same float32 W, applied and differentiated on bf16 tensor cores (layers/dense_bf16.py)."""

    @staticmethod
    def forward(ctx, U, bias, layer, A, Bm, G, H):
        W, ws, status, max_terms, slots, Gc, Hc = _ldr_build_weight(layer, U.device, A, Bm, G, H)
        x = D.staged(U)
        y, Wtb = D.forward(layer, W, x, bias, keep_wt=ctx.needs_input_grad[0])
        ctx.max_terms, ctx.slots, ctx.has_bias = max_terms, slots, bias is not None
        ctx.save_for_backward(x, ws, status, Wtb, A, Bm, Gc, Hc)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        x, ws, status, Wtb, A, Bm, G, H = ctx.saved_tensors
        n = G.shape[0]
        gy = D.staged(grad_y)
        grad_x = D.input_grad(Wtb, gy) if ctx.needs_input_grad[0] else None
        dW = torch.zeros((n, n), dtype=torch.float32, device=x.device)
        gbias = torch.zeros(n, dtype=torch.float32, device=x.device) if ctx.has_bias else None
        D.weight_grad(x, gy, dW, gbias)
        gAs, gBs, gG, gH = _ldr_param_grads(dW, ctx.slots, ws, ctx.max_terms, status, A, Bm, G, H)
        return grad_x, gbias, None, gAs, gBs, gG, gH


class LDRLayer(StructuredLayer):
    def __init__(self, input_dim: int, output_dim: int, nb_params_share: float, use_bias=True, initial_weight_matrix=None,
                 initial_bias=None, initial_representation_matrices=None):
        super(LDRLayer, self).__init__(input_dim=input_dim, output_dim=output_dim, nb_params_share=nb_params_share, use_bias=use_bias,
                                       initial_weight_matrix=initial_weight_matrix, initial_bias=initial_bias)
        assert input_dim == output_dim, "The LDR Layer is only implemented for square weight matrices (i.e. when the number of inputs equals the number of outputs)"
        assert initial_weight_matrix is None or initial_representation_matrices is None, "Either pass an initial weight matrix or initial representation matrices - not both"
        if initial_representation_matrices is not None:
            assert len(initial_representation_matrices) == 4, "Expect the length of the list of initial representation matrices to be 4"
            for representation_matrix in initial_representation_matrices:
                assert torch.is_tensor(representation_matrix), "Expect all representation matrices to be given as torch.tensor"

        self.input_dim = input_dim
        self.target_mat_shape = (self.output_dim, input_dim)
        max_nb_parameters = int(nb_params_share * input_dim * self.output_dim)
        displacement_rank = get_max_ld_rank_wrt_max_nb_free_parameters(max_nb_free_parameters=max_nb_parameters, target_shape_mat=self.target_mat_shape)

        if displacement_rank < 0:
            self.representation_matrices = None
            self.fake_optim_param = nn.Parameter(get_random_glorot_uniform_matrix_torch((1, 1)))
        else:
            if initial_representation_matrices is not None:
                representation_matrices = pickle.loads(pickle.dumps(initial_representation_matrices))
            elif initial_weight_matrix is not None:
                raise NotImplementedError(
                    "LDRLayer: fitting the representation to a dense matrix is the reference's init-time LDRApproximator "
                    "(torch-SGD with restarts, approximators/ldr_approximator.py:61-139), out of scope here (SURVEY.md section 2); "
                    "pass initial_representation_matrices=...")
            else:
                representation_matrices = init_representation_matrices_torch(shape=self.target_mat_shape, displacement_rank=displacement_rank)
            self.representation_matrices = nn.ParameterList([nn.Parameter(m.detach()) for m in representation_matrices])

    def _slots(self, A, Bm):
        cache = self.__dict__.get("_dev_slots")
        key = (A._indices().data_ptr(), A._nnz(), Bm._indices().data_ptr(), Bm._nnz(), str(A.device))
        if cache is None or cache[0] != key:
            n = self.output_dim
            cache = (key, (band_slots(A._indices(), n), band_slots(Bm._indices(), n)))
            self.__dict__["_dev_slots"] = cache
        return cache[1]

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop("_dev_slots", None)
        state.pop("_dev_W_bf16", None)
        return state

    def forward(self, U):
        if self.representation_matrices is None:
            return torch.zeros((U.shape[0], self.output_dim), device=U.device)   # reference ldr_layer.py:51-52
        self._require_cuda(U, "LDRLayer.forward")
        assert U.dim() == 2 and U.shape[1] == self.input_dim, "LDRLayer expects a (batch, input_dim) input"
        if U.dtype == torch.bfloat16:     # bf16 output, float32 / float64 parameters and gradients
            return _LDRBF16Function.apply(U, self.bias if self.use_bias else None, self, *self.representation_matrices)
        if U.dtype != torch.float32:
            U = U.float()
        if U.stride(1) != 1:
            U = U.contiguous()
        return _LDRFunction.apply(U, self.bias if self.use_bias else None, self, *self.representation_matrices)

    def get_nb_parameters(self) -> int:
        # the reference's version reads non-existent attributes (ldr_layer.py:67; SURVEY.md "smaller bugs"):
        # return what it evidently means -- the free parameters of the representation plus the bias.
        if self.representation_matrices is None:
            return 0
        res = sum(int(p._nnz()) if p.is_sparse else int(p.numel()) for p in self.representation_matrices)
        if self.use_bias:
            res += torch.numel(self.bias)
        return int(res)
