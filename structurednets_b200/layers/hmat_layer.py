"""Hierarchical-matrix layer on B200.  Drop-in for ``structurednets.layers.hmat_layer.HMatLayer``
(reference layers/hmat_layer.py:12-52): same constructor, a ``ModuleList`` ``hmatrix_components`` of
leaves with parameters ``left_lr`` / ``right_lr`` (state_dict keys
``bias, hmatrix_components.{i}.left_lr, hmatrix_components.{i}.right_lr``), leaves with rank 0 dropped.
Forward/backward run in csrc/hmat.cu through ``sn_hmat_forward`` / ``sn_hmat_backward``.
"""
import os

import numpy as np
import torch
import torch.nn as nn

from structurednets_b200 import _lib
from structurednets_b200.layers import dense_bf16 as D
from structurednets_b200.hmatrix.hmatrix import BlockClusterTree, HMatrix, HMatrixComponent, TreeElement, approximate_hmatrix
from structurednets_b200.layers.flat_params import FlatParamsMixin
from structurednets_b200.layers.layer_helpers import get_random_glorot_uniform_matrix
from structurednets_b200.layers.structured_layer import StructuredLayer


class _HMatFunction(torch.autograd.Function):
    """Leaf-by-leaf CUDA-core kernels (csrc/hmat.cu: sn_hmat_forward / sn_hmat_backward); kept for matrices too large to densify.
    ``anchor`` is passed when some parameter takes a gradient; a backward that only returns ``grad_x`` leaves the flat gradient
    buffer alone."""

    @staticmethod
    def forward(ctx, U, anchor, layer):
        B = U.shape[0]
        table = layer._leaf_table(U.device)
        flat = layer.flat_parameters()
        y = torch.empty((B, layer.output_dim), dtype=torch.float32, device=U.device)
        rc = _lib.lib().sn_hmat_forward(_lib.ptr(table), layer._nleaves, _lib.ptr(flat), _lib.ptr(U), U.stride(0), _lib.ptr(y),
                                        y.stride(0), _lib.ptr(layer.bias if layer.use_bias else None), B, layer.input_dim,
                                        layer.output_dim, _lib.stream_ptr())
        _lib.check(rc, "sn_hmat_forward")
        ctx.layer = layer
        ctx.param_grad = anchor is not None
        ctx.save_for_backward(U, table)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        layer = ctx.layer
        U, table = ctx.saved_tensors
        grad_y = grad_y.contiguous().float()
        grad_x = torch.empty_like(U) if ctx.needs_input_grad[0] else None
        g = layer._prepare_grad_accumulation() if ctx.param_grad else None
        gb = g[:layer.output_dim] if (g is not None and layer.use_bias and layer.bias.requires_grad) else None
        rc = _lib.lib().sn_hmat_backward(_lib.ptr(table), layer._nleaves, _lib.ptr(layer.flat_parameters()), _lib.ptr(U), U.stride(0),
                                         _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(g), _lib.ptr(gb), _lib.ptr(grad_x),
                                         grad_x.stride(0) if grad_x is not None else 0, U.shape[0], layer.input_dim, layer.output_dim,
                                         _lib.stream_ptr())
        _lib.check(rc, "sn_hmat_backward")
        return grad_x, None, None


class _HMatDenseFunction(torch.autograd.Function):
    """Dense-block path: the leaves are multiplied out into one dense matrix (sn_hmat_build_dense), the batch goes through the
    tensor-core GEMMs shared with the LDR / TL layers (sn_dense_apply, sn_dense_weight_grad) and the dense gradient is projected
    back onto the leaf factors (sn_hmat_project_grad)."""

    @staticmethod
    def forward(ctx, U, anchor, layer):
        B = U.shape[0]
        L = _lib.lib()
        table = layer._leaf_table(U.device)
        flat = layer.flat_parameters()
        W = layer._dense_buffer("_dev_W", U.device)
        slabs = layer._slab_table(U.device)
        _lib.check(L.sn_hmat_build_dense(_lib.ptr(table), layer._nleaves, layer._max_leaf_rows, _lib.ptr(slabs), slabs.numel() // 2, _lib.ptr(flat),
                                         _lib.ptr(W), layer.output_dim, layer.input_dim, _lib.stream_ptr()), "sn_hmat_build_dense")
        y = torch.empty((B, layer.output_dim), dtype=torch.float32, device=U.device)
        _lib.check(L.sn_dense_apply(_lib.ptr(W), layer.output_dim, layer.input_dim, _lib.ptr(U), U.stride(0), _lib.ptr(y), y.stride(0),
                                    _lib.ptr(layer.bias if layer.use_bias else None), B, _lib.stream_ptr()), "sn_dense_apply")
        ctx.layer = layer
        ctx.save_for_backward(U, table)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        layer = ctx.layer
        U, table = ctx.saved_tensors
        grad_y = grad_y.contiguous().float()
        L = _lib.lib()
        grad_x = None
        if ctx.needs_input_grad[0]:
            # the dense W of this layer's last forward (a layer-wide buffer: forward -> backward without another forward in between)
            W = layer._dense_buffer("_dev_W", U.device)
            grad_x = torch.empty_like(U)
            _lib.check(L.sn_dense_input_grad(_lib.ptr(W), layer.output_dim, layer.input_dim, _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(grad_x),
                                             grad_x.stride(0), U.shape[0], _lib.stream_ptr()), "sn_dense_input_grad")
        g = layer._prepare_grad_accumulation()
        gb = g[:layer.output_dim] if (layer.use_bias and layer.bias.requires_grad) else None
        dW = layer._dense_buffer("_dev_dW", U.device)
        dW.zero_()
        _lib.check(L.sn_dense_weight_grad(_lib.ptr(U), U.stride(0), _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(dW), layer.output_dim,
                                          layer.input_dim, _lib.ptr(gb), U.shape[0], _lib.stream_ptr()), "sn_dense_weight_grad")
        slabs = layer._slab_table(U.device)
        _lib.check(L.sn_hmat_project_grad(_lib.ptr(table), layer._nleaves, _lib.ptr(slabs), slabs.numel() // 2, _lib.ptr(layer.flat_parameters()),
                                          _lib.ptr(dW), layer.output_dim, layer.input_dim, _lib.ptr(g), _lib.stream_ptr()), "sn_hmat_project_grad")
        return grad_x, None, None


class _HMatDenseBF16Function(torch.autograd.Function):
    """bfloat16 features on the dense-block path: the same float32 W (sn_hmat_build_dense) and projection (sn_hmat_project_grad),
    the batch GEMMs on bf16 tensor cores (layers/dense_bf16.py).  Like the float32 path, the projection reads the layer's current
    parameters: forward -> backward without a parameter update in between."""

    @staticmethod
    def forward(ctx, U, anchor, layer):
        L = _lib.lib()
        table = layer._leaf_table(U.device)
        W = layer._dense_buffer("_dev_W", U.device)
        slabs = layer._slab_table(U.device)
        _lib.check(L.sn_hmat_build_dense(_lib.ptr(table), layer._nleaves, layer._max_leaf_rows, _lib.ptr(slabs), slabs.numel() // 2,
                                         _lib.ptr(layer.flat_parameters()), _lib.ptr(W), layer.output_dim, layer.input_dim, _lib.stream_ptr()),
                   "sn_hmat_build_dense")
        x = D.staged(U)
        y, Wtb = D.forward(layer, W, x, layer.bias if layer.use_bias else None, keep_wt=ctx.needs_input_grad[0])
        ctx.layer = layer
        ctx.save_for_backward(x, table, Wtb)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        layer = ctx.layer
        x, table, Wtb = ctx.saved_tensors
        gy = D.staged(grad_y)
        grad_x = D.input_grad(Wtb, gy) if ctx.needs_input_grad[0] else None
        g = layer._prepare_grad_accumulation()
        gb = g[:layer.output_dim] if (layer.use_bias and layer.bias.requires_grad) else None
        dW = layer._dense_buffer("_dev_dW", x.device)
        dW.zero_()
        D.weight_grad(x, gy, dW, gb)
        slabs = layer._slab_table(x.device)
        _lib.check(_lib.lib().sn_hmat_project_grad(_lib.ptr(table), layer._nleaves, _lib.ptr(slabs), slabs.numel() // 2,
                                                   _lib.ptr(layer.flat_parameters()), _lib.ptr(dW), layer.output_dim, layer.input_dim, _lib.ptr(g),
                                                   _lib.stream_ptr()), "sn_hmat_project_grad")
        return grad_x, None, None


class HMatLayer(FlatParamsMixin, StructuredLayer):
    def __init__(self, input_dim: int, output_dim: int, nb_params_share: float, use_bias=True, initial_weight_matrix=None,
                 initial_bias=None, eta=0.5, initial_hmatrix=None, use_gpu=False):
        super(HMatLayer, self).__init__(input_dim=input_dim, output_dim=output_dim, nb_params_share=nb_params_share, use_bias=use_bias,
                                        initial_weight_matrix=initial_weight_matrix, initial_bias=initial_bias)
        assert initial_weight_matrix is None or initial_hmatrix is None, "You can either pass an initial hmatrix or an initial weight matrix to be used as starting point fo the HMatrixLayer"

        if initial_hmatrix is not None:
            self.hmatrix = initial_hmatrix.clone()
        else:
            if initial_weight_matrix is None:
                initial_weight_matrix = get_random_glorot_uniform_matrix((output_dim, input_dim))
            # use_gpu (reference hmat_layer.py:13,36-37: "put the scratch tensors on the GPU") also moves the per-leaf SVDs of the
            # initialisation to the GPU, batched by leaf shape
            svd_device = "cuda" if (use_gpu and torch.cuda.is_available()) else None
            self.hmatrix = approximate_hmatrix(initial_weight_matrix, nb_params_share=nb_params_share, eta=eta, device=svd_device)

        self.input_dim = input_dim
        components = [c for c in self.hmatrix.get_all_hmatrix_components() if c.are_low_rank_components_set()]
        # re-wrap foreign (e.g. reference) component objects so parameters are float32 leaves we own
        own = []
        for c in components:
            if isinstance(c, HMatrixComponent):
                own.append(c)
            else:
                own.append(HMatrixComponent(c.row_range, c.col_range, c.left_lr.detach(), c.right_lr.detach()))
        self.hmatrix_components = nn.ModuleList(own)
        self.use_gpu = use_gpu
        self._nleaves = len(own)
        self._max_leaf_rows = max([len(c.row_range) for c in own], default=1)
        self._flatten_parameters()

    # ---- pickling: the tree in ``self.hmatrix`` references the same leaf modules as ``hmatrix_components``; pickled as it is, every
    # leaf parameter (a view of the flat buffer) would carry the whole flat storage.  Only the tree's ranges are stored, the leaves
    # are re-bound to ``hmatrix_components`` on load, so ``hmatrix.to_dense()`` keeps tracking the trained parameters.
    def __getstate__(self):
        state = super().__getstate__()
        hm = state.get("hmatrix")
        if isinstance(hm, HMatrix) and isinstance(hm.block_cluster_tree, BlockClusterTree):
            index = {id(c): i for i, c in enumerate(self.hmatrix_components)}

            def skeleton(el):
                if el.is_leaf():
                    return (el.row_range, el.col_range, index.get(id(el.hmatrix_component), -1))
                return (el.row_range, el.col_range, [skeleton(ch) for ch in el.children])
            state["hmatrix"] = None
            state["_hmatrix_skeleton"] = (skeleton(hm.block_cluster_tree.root), getattr(hm, "shape", None))
        return state

    def __setstate__(self, state):
        state = dict(state)
        sk = state.pop("_hmatrix_skeleton", None)
        super().__setstate__(state)
        if sk is not None:
            comps = list(self.hmatrix_components)

            def rebuild(node):
                rows, cols, rest = node
                el = TreeElement(None, rows, cols)
                if isinstance(rest, list):
                    el.children = [rebuild(ch) for ch in rest]
                elif rest >= 0:
                    el.hmatrix_component = comps[rest]
                return el
            self.hmatrix = HMatrix(BlockClusterTree(rebuild(sk[0])), shape=sk[1])

    DENSE_PATH_MAX_ELEMENTS = 1 << 26   # dense (out x in) fp32 copies of at most 256 MB each

    def _on_reflatten(self):
        self.__dict__["_dev_table"] = None
        self.__dict__["_dev_slabs"] = None
        self.__dict__["_dev_W"] = None
        self.__dict__["_dev_dW"] = None

    def _dense_buffer(self, key, device):
        t = self.__dict__.get(key)
        if t is None or t.device != device:
            t = torch.empty((self.output_dim, self.input_dim), dtype=torch.float32, device=device)
            self.__dict__[key] = t
        return t

    def _use_dense_path(self) -> bool:
        mode = os.environ.get("SNB200_HMAT_PATH", "auto")
        if mode == "leaf":
            return False
        return mode == "dense" or self.output_dim * self.input_dim <= self.DENSE_PATH_MAX_ELEMENTS

    def build_leaf_table(self) -> np.ndarray:
        """(nleaves, 8) int32: row_start, rows, col_start, cols, rank, off_left, off_right, 0 (see csrc/hmat.cu)."""
        self._ensure_flat()
        by_id = {id(p): o for p, o in zip(self._flat_param_list(), self.__dict__["_flat_offsets"])}
        tab = np.zeros((max(self._nleaves, 1), 8), dtype=np.int32)
        for i, c in enumerate(self.hmatrix_components):
            k = c.left_lr.shape[1]
            assert c.left_lr.shape[0] == len(c.row_range) and c.right_lr.shape[1] == len(c.col_range) and c.right_lr.shape[0] == k
            assert c.row_range.stop <= self.output_dim and c.col_range.stop <= self.input_dim
            tab[i] = [c.row_range.start, len(c.row_range), c.col_range.start, len(c.col_range), k, by_id[id(c.left_lr)], by_id[id(c.right_lr)], 0]
        # largest leaves first: better balance of the per-warp round-robin (order does not change the result
        # beyond fp32 summation order)
        order = np.argsort(-(tab[:, 4].astype(np.int64) * (tab[:, 1] + tab[:, 3])), kind="stable")
        return tab[order]

    def _slab_table(self, device):
        """(leaf index in the device leaf table, first row) per 32 rows of every leaf: the work list of sn_hmat_project_grad."""
        t = self.__dict__.get("_dev_slabs")
        if t is None or t.device != device:
            tab = self.build_leaf_table()
            pairs = [(i, r0) for i in range(self._nleaves) for r0 in range(0, int(tab[i, 1]), 32)]
            t = torch.tensor(np.asarray(pairs, dtype=np.int32).reshape(-1), device=device)
            self.__dict__["_dev_slabs"] = t
        return t

    def _leaf_table(self, device):
        self._ensure_flat()
        t = self.__dict__.get("_dev_table")
        if t is None or t.device != device:
            t = torch.from_numpy(self.build_leaf_table().reshape(-1)).to(device)
            self.__dict__["_dev_table"] = t
        return t

    def forward(self, U):
        self._require_cuda(U, "HMatLayer.forward")
        assert U.dim() == 2 and U.shape[1] == self.input_dim, "HMatLayer expects a (batch, input_dim) input"
        self._ensure_flat()
        if U.dtype == torch.bfloat16 and self._use_dense_path():   # bf16 output, float32 parameters and gradients
            fn = _HMatDenseBF16Function
        else:
            fn = _HMatDenseFunction if self._use_dense_path() else _HMatFunction
            if U.dtype != torch.float32:
                U = U.float()
            if U.stride(1) != 1:
                U = U.contiguous()
        anchor = self.__dict__.get("_dev_anchor")
        if anchor is None or anchor.device != U.device:
            anchor = torch.zeros(1, device=U.device, requires_grad=True)
            self.__dict__["_dev_anchor"] = anchor
        needs = torch.is_grad_enabled() and self._nleaves > 0
        if fn is _HMatFunction:
            # the leaf path computes parameter gradients only when some parameter takes one (SSSLayer decides the same way)
            needs = needs and any(p.requires_grad for p in self._flat_param_list())
        return fn.apply(U, anchor if needs else None, self)

    def get_nb_parameters(self) -> int:
        return self.hmatrix.get_nb_params()
