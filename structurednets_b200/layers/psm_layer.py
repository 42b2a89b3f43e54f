"""Product-of-sparse-matrices layer on B200.  Drop-in for ``structurednets.layers.psm_layer.PSMLayer``
(reference layers/psm_layer.py:13-80): same constructor (note the reference's positional order
``input_dim, output_dim, use_bias, nb_params_share, ...``), a ``ParameterList`` ``sparse_matrices`` of
float32 sparse-COO parameters built exactly like ``scipy_csr_to_torch`` (psm_layer.py:30-34) and sparse
gradients on the same pattern, so the "SGD only" behaviour of the reference is unchanged.

Factor order: the intended chain W = S0 S1 ... S(n-1) (psm_approximator.py:96-105).  The reference's
forward applies ``[-1], [0], [1], ...`` (psm_layer.py:52-54), which equals the intended order for <= 2
factors and is a shape error / wrong product for >= 3 (SURVEY.md finding F2).
"""
import ctypes

import numpy as np
import scipy.sparse
import torch
import torch.nn as nn

from structurednets_b200 import _lib
from structurednets_b200.layers import dense_bf16 as D
from structurednets_b200.layers.layer_helpers import get_random_glorot_uniform_matrix
from structurednets_b200.layers.structured_layer import StructuredLayer


def _sliced_ell(rows: np.ndarray, cols: np.ndarray, nr: int):
    """Sliced-ELL arrangement of a COO pattern (csrc/psm.cu): rows sorted by length, slices of 32 rows, entry j of the 32 rows
    of a slice contiguous.  Returns numpy arrays rowmap, slice_off, col (uint16), src (COO index or -1)."""
    nnz = len(rows)
    counts = np.bincount(rows, minlength=nr).astype(np.int64)
    order = np.argsort(-counts, kind="stable")
    nslices = (nr + 31) // 32
    rowmap = np.full(nslices * 32, -1, dtype=np.int32)
    rowmap[:nr] = order
    pos_of_row = np.empty(nr, dtype=np.int64)
    pos_of_row[order] = np.arange(nr)
    padded = np.zeros(nslices * 32, dtype=np.int64)
    padded[:nr] = counts[order]
    slice_len = padded.reshape(nslices, 32).max(axis=1)
    slice_off = np.concatenate([[0], np.cumsum(slice_len * 32)]).astype(np.int64)
    total = int(slice_off[-1])
    perm = np.argsort(rows, kind="stable")
    r_sorted = rows[perm]
    start = np.cumsum(counts) - counts
    j = np.arange(nnz) - start[r_sorted]
    p = pos_of_row[r_sorted]
    dest = slice_off[p // 32] + j * 32 + (p % 32)
    col = np.zeros(max(total, 1), dtype=np.uint16)
    src = np.full(max(total, 1), -1, dtype=np.int32)
    col[dest] = cols[perm].astype(np.uint16)
    src[dest] = perm.astype(np.int32)
    return dict(nslices=nslices, total=total, rowmap=rowmap, slice_off=slice_off.astype(np.int32), col=col, src=src)


def _pattern(p: torch.Tensor):
    """Sliced-ELL forms of an (uncoalesced) sparse-COO pattern and of its transpose, plus the per-call scratch the kernels need;
    cached per indices storage (built on the host once: the pattern is static)."""
    idx = p._indices()
    dev = idx.device
    rows, cols = idx[0].cpu().numpy().astype(np.int64), idx[1].cpu().numpy().astype(np.int64)
    nr, nc = p.shape
    assert nr <= 65535 and nc <= 65535, "PSMLayer: factor dimensions above 65535 are not supported by the CUDA path"
    out = dict(key=(idx.data_ptr(), idx.shape[1], str(dev)))
    for name, e in (("fwd", _sliced_ell(rows, cols, nr)), ("tr", _sliced_ell(cols, rows, nc))):
        d = dict(nslices=e["nslices"], total=e["total"])
        d["rowmap"] = torch.from_numpy(e["rowmap"]).to(dev)
        d["slice_off"] = torch.from_numpy(e["slice_off"]).to(dev)
        d["col"] = torch.from_numpy(e["col"].view(np.int16)).to(dev)
        d["src"] = torch.from_numpy(e["src"]).to(dev)
        d["val"] = torch.zeros(max(e["total"], 1), dtype=torch.float32, device=dev)
        out[name] = d
    out["grad_packed"] = torch.zeros(max(out["fwd"]["total"], 1), dtype=torch.float32, device=dev)
    return out


def _dense_pattern(p: torch.Tensor):
    """CSR / CSC / COO (int32) forms of a sparse-COO pattern for the dense-product path (csrc/psm.cu), built once on the host."""
    idx = p._indices()
    dev = idx.device
    rows, cols = idx[0].cpu().numpy().astype(np.int64), idx[1].cpu().numpy().astype(np.int64)
    nr, nc = p.shape
    out = dict(key=(idx.data_ptr(), idx.shape[1], str(dev)))
    for name, major, minor, n in (("csr", rows, cols, nr), ("csc", cols, rows, nc)):
        order = np.argsort(major, kind="stable")
        ptr = np.concatenate([[0], np.cumsum(np.bincount(major, minlength=n))]).astype(np.int32)
        out[name + "_ptr"] = torch.from_numpy(ptr).to(dev)
        out[name + "_idx"] = torch.from_numpy(minor[order].astype(np.int32)).to(dev)
        out[name + "_src"] = torch.from_numpy(order.astype(np.int32)).to(dev)
    out["coo_row"] = torch.from_numpy(rows.astype(np.int32)).to(dev)
    out["coo_col"] = torch.from_numpy(cols.astype(np.int32)).to(dev)
    return out


def _dense_factor_array(patterns, params, gvals):
    arr = (_lib.SnPsmDenseFactor * len(params))()
    for k, (pat, p) in enumerate(zip(patterns, params)):
        f = arr[k]
        f.rows, f.cols, f.nnz = int(p.shape[0]), int(p.shape[1]), int(p._nnz())
        for n in ("csr_ptr", "csr_idx", "csr_src", "csc_ptr", "csc_idx", "csc_src", "coo_row", "coo_col"):
            setattr(f, n, pat[n].data_ptr())
        f.vals = p._values().data_ptr()
        f.grad_vals = gvals[k].data_ptr() if gvals is not None else None
    return arr


class _PSMDenseFunction(torch.autograd.Function):
    """Large-batch path: the factors are multiplied out once per call, the batch goes through the tensor-core GEMMs."""

    @staticmethod
    def forward(ctx, U, bias, layer, *factors):
        B = U.shape[0]
        patterns = layer._dense_patterns(factors)
        assert all(p._values().dtype == torch.float32 and p._values().is_contiguous() for p in factors)
        arr = _dense_factor_array(patterns, factors, None)
        L = _lib.lib()
        prefix = torch.empty(L.sn_psm_dense_prefix_floats(arr, len(factors), layer.output_dim), dtype=torch.float32, device=U.device)
        y = torch.empty((B, layer.output_dim), dtype=torch.float32, device=U.device)
        rc = L.sn_psm_dense_forward(arr, len(factors), _lib.ptr(U), U.stride(0), _lib.ptr(y), y.stride(0), _lib.ptr(bias), _lib.ptr(prefix), B,
                                    layer.input_dim, layer.output_dim, _lib.stream_ptr())
        _lib.check(rc, "sn_psm_dense_forward")
        ctx.layer, ctx.patterns, ctx.has_bias = layer, patterns, bias is not None
        ctx.save_for_backward(U, prefix, *factors)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        U, prefix, *factors = ctx.saved_tensors
        layer = ctx.layer
        grad_y = grad_y.contiguous().float()
        gvals = [torch.zeros(p._nnz(), dtype=torch.float32, device=U.device) for p in factors]
        gbias = torch.zeros(layer.output_dim, dtype=torch.float32, device=U.device) if ctx.has_bias else None
        arr = _dense_factor_array(ctx.patterns, factors, gvals)
        L = _lib.lib()
        work = torch.empty(L.sn_psm_dense_backward_floats(arr, len(factors), layer.output_dim), dtype=torch.float32, device=U.device)
        rc = L.sn_psm_dense_backward(arr, len(factors), _lib.ptr(U), U.stride(0), _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(prefix),
                                     _lib.ptr(work), _lib.ptr(gbias), U.shape[0], layer.input_dim, layer.output_dim, _lib.stream_ptr())
        _lib.check(rc, "sn_psm_dense_backward")
        grad_x = None
        if ctx.needs_input_grad[0]:
            grad_x = torch.empty_like(U)
            _lib.check(L.sn_psm_dense_input_grad(arr, len(factors), _lib.ptr(prefix), _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(grad_x),
                                                 grad_x.stride(0), U.shape[0], layer.input_dim, layer.output_dim, _lib.stream_ptr()), "sn_psm_dense_input_grad")
        gf = [torch.sparse_coo_tensor(p._indices(), g, p.shape) for p, g in zip(factors, gvals)]
        return (grad_x, gbias, None, *gf)


class _PSMDenseBF16Function(torch.autograd.Function):
    """bfloat16 features: the dense-product path's prefix products and projection, the batch GEMMs on bf16 tensor cores
    (sn_psm_dense_forward_bf16 / sn_psm_dense_backward_bf16, layers/dense_bf16.py)."""

    @staticmethod
    def forward(ctx, U, bias, layer, *factors):
        patterns = layer._dense_patterns(factors)
        assert all(p._values().dtype == torch.float32 and p._values().is_contiguous() for p in factors)
        arr = _dense_factor_array(patterns, factors, None)
        L = _lib.lib()
        x = D.staged(U)
        B, dev = x.shape[0], x.device
        prefix = torch.empty(L.sn_psm_dense_prefix_floats(arr, len(factors), layer.output_dim), dtype=torch.float32, device=dev)
        Wb = D.weight_buffer(layer, layer.output_dim, layer.input_dim, dev)
        Wtb = torch.empty((layer.input_dim, D.pad8(layer.output_dim)), dtype=torch.bfloat16, device=dev) if ctx.needs_input_grad[0] else None
        y = D.empty_rows(B, layer.output_dim, dev)
        rc = L.sn_psm_dense_forward_bf16(arr, len(factors), _lib.ptr(x), x.stride(0), _lib.ptr(y), y.stride(0), _lib.ptr(bias), _lib.ptr(prefix),
                                         _lib.ptr(Wb), Wb.stride(0), _lib.ptr(Wtb), Wtb.stride(0) if Wtb is not None else 0, B, layer.input_dim,
                                         layer.output_dim, _lib.stream_ptr())
        _lib.check(rc, "sn_psm_dense_forward_bf16")
        ctx.layer, ctx.patterns, ctx.has_bias = layer, patterns, bias is not None
        ctx.save_for_backward(x, prefix, Wtb, *factors)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        x, prefix, Wtb, *factors = ctx.saved_tensors
        layer = ctx.layer
        gy = D.staged(grad_y)
        gvals = [torch.zeros(p._nnz(), dtype=torch.float32, device=x.device) for p in factors]
        gbias = torch.zeros(layer.output_dim, dtype=torch.float32, device=x.device) if ctx.has_bias else None
        arr = _dense_factor_array(ctx.patterns, factors, gvals)
        L = _lib.lib()
        work = torch.empty(L.sn_psm_dense_backward_floats(arr, len(factors), layer.output_dim), dtype=torch.float32, device=x.device)
        rc = L.sn_psm_dense_backward_bf16(arr, len(factors), _lib.ptr(x), x.stride(0), _lib.ptr(gy), gy.stride(0), _lib.ptr(prefix), _lib.ptr(work),
                                          _lib.ptr(gbias), x.shape[0], layer.input_dim, layer.output_dim, _lib.stream_ptr())
        _lib.check(rc, "sn_psm_dense_backward_bf16")
        grad_x = D.input_grad(Wtb, gy) if ctx.needs_input_grad[0] else None
        gf = [torch.sparse_coo_tensor(p._indices(), g, p.shape) for p, g in zip(factors, gvals)]
        return (grad_x, gbias, None, *gf)


def _factor_array(patterns, params, gvals):
    arr = (_lib.SnPsmFactor * len(params))()
    for k, (pat, p) in enumerate(zip(patterns, params)):
        f = arr[k]
        f.rows, f.cols, f.nnz = int(p.shape[0]), int(p.shape[1]), int(p._nnz())
        for name in ("fwd", "tr"):
            e, d = getattr(f, name), pat[name]
            e.nslices, e.total = d["nslices"], d["total"]
            e.rowmap, e.slice_off, e.col, e.src = d["rowmap"].data_ptr(), d["slice_off"].data_ptr(), d["col"].data_ptr(), d["src"].data_ptr()
        f.vals = p._values().data_ptr()
        f.val_fwd, f.val_tr = pat["fwd"]["val"].data_ptr(), pat["tr"]["val"].data_ptr()
        f.grad_packed = pat["grad_packed"].data_ptr() if gvals is not None else None
        f.grad_vals = gvals[k].data_ptr() if gvals is not None else None
    return arr


class _PSMFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, U, bias, layer, *factors):
        B = U.shape[0]
        patterns = layer._patterns(factors)
        vals = [p._values() for p in factors]
        assert all(v.dtype == torch.float32 and v.is_contiguous() for v in vals)
        arr = _factor_array(patterns, factors, None)
        y = torch.empty((B, layer.output_dim), dtype=torch.float32, device=U.device)
        # the inputs of the inner factors are kept for the backward (no recomputation) when anything takes a gradient
        needs = any(ctx.needs_input_grad[3:]) or (bias is not None and ctx.needs_input_grad[1])
        acts = None
        if needs and len(factors) > 1:
            acts = torch.empty(int(_lib.lib().sn_psm_acts_floats(arr, len(factors), B)), dtype=torch.float32, device=U.device)
        rc = _lib.lib().sn_psm_forward(arr, len(factors), _lib.ptr(U), U.stride(0), _lib.ptr(y), y.stride(0), _lib.ptr(bias), _lib.ptr(acts), B,
                                       layer.input_dim, layer.output_dim, _lib.stream_ptr())
        _lib.check(rc, "sn_psm_forward")
        ctx.layer, ctx.patterns, ctx.has_bias, ctx.has_acts = layer, patterns, bias is not None, acts is not None
        ctx.save_for_backward(U, acts if acts is not None else U.new_empty(0), *factors)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        U, acts, *factors = ctx.saved_tensors
        acts = acts if ctx.has_acts else None
        layer = ctx.layer
        grad_y = grad_y.contiguous().float()
        grad_x = torch.empty_like(U) if ctx.needs_input_grad[0] else None
        # the factor gradients are computed when a factor takes one (or when nothing else would run: a bias-only backward)
        param_grad = any(ctx.needs_input_grad[3:]) or grad_x is None
        gvals = [torch.zeros(p._nnz(), dtype=torch.float32, device=U.device) for p in factors] if param_grad else None
        # (without grad_x, param_grad holds and the bias gradient is formed as it always was)
        gbias = torch.zeros(layer.output_dim, dtype=torch.float32, device=U.device) if ctx.has_bias and (param_grad or ctx.needs_input_grad[1]) else None
        arr = _factor_array(ctx.patterns, factors, gvals)
        rc = _lib.lib().sn_psm_backward(arr, len(factors), _lib.ptr(U), U.stride(0), _lib.ptr(grad_y), grad_y.stride(0), _lib.ptr(acts), _lib.ptr(gbias),
                                        _lib.ptr(grad_x), grad_x.stride(0) if grad_x is not None else 0, U.shape[0], layer.input_dim,
                                        layer.output_dim, _lib.stream_ptr())
        _lib.check(rc, "sn_psm_backward")
        # sparse gradients on the parameters' own (uncoalesced) pattern, like autograd's to_dense backward
        gf = [torch.sparse_coo_tensor(p._indices(), g, p.shape) if need else None
              for p, g, need in zip(factors, gvals or [None] * len(factors), ctx.needs_input_grad[3:])]
        return (grad_x, gbias, None, *gf)


class PSMLayer(StructuredLayer):
    # NOTE (reference psm_layer.py:14-15): sparse weight matrices -> sparse gradients -> train with SGD, not Adam.
    def __init__(self, input_dim: int, output_dim: int, use_bias=True, nb_params_share=None, initial_weight_matrix=None,
                 initial_bias=None, sparse_matrices=None):
        super(PSMLayer, self).__init__(input_dim=input_dim, output_dim=output_dim, nb_params_share=nb_params_share, use_bias=use_bias,
                                       initial_weight_matrix=initial_weight_matrix, initial_bias=initial_bias)
        assert nb_params_share is not None or sparse_matrices is not None, "Need to pass the nb_params_share or an initial sparse matrices configuration"
        assert sparse_matrices is None or initial_weight_matrix is None, "Can either pass an initial weight matrix or an initial sparse matrices configuration"

        if sparse_matrices is None:
            if initial_weight_matrix is None:
                initial_weight_matrix = get_random_glorot_uniform_matrix((output_dim, input_dim))
            sparse_matrices = _factorize(initial_weight_matrix, nb_params_share)

        self.input_dim = input_dim
        self.sparse_matrices = nn.ParameterList([self.scipy_csr_to_torch(mat) for mat in sparse_matrices])
        self._base_nnz = [int(p._nnz()) for p in self.sparse_matrices]
        shapes = [tuple(p.shape) for p in self.sparse_matrices]
        assert shapes[0][0] == output_dim and shapes[-1][1] == input_dim, "The sparse factors do not map input_dim -> output_dim"
        for a, b in zip(shapes[:-1], shapes[1:]):
            assert a[1] == b[0], "Consecutive sparse factors cannot be multiplied: " + str(shapes)

    def scipy_csr_to_torch(self, mat) -> torch.Tensor:
        """Same construction as the reference (psm_layer.py:30-34): transpose of the COO with swapped indices."""
        coo_mat = scipy.sparse.coo_matrix(mat)
        idx = torch.tensor(np.stack([coo_mat.col, coo_mat.row]).astype(np.int64))
        res = torch.transpose(torch.sparse_coo_tensor(idx, torch.tensor(coo_mat.data), (coo_mat.shape[1], coo_mat.shape[0])).float(), 0, 1)
        res.requires_grad_(True)
        return nn.Parameter(res)

    def _patterns(self, factors):
        cache = self.__dict__.setdefault("_dev_patterns", {})
        out = []
        for k, p in enumerate(factors):
            idx = p._indices()
            key = (idx.data_ptr(), idx.shape[1], str(idx.device))
            pat = cache.get(k)
            if pat is None or pat["key"] != key:
                pat = _pattern(p)
                cache[k] = pat
            out.append(pat)
        return out

    def _dense_patterns(self, factors):
        cache = self.__dict__.setdefault("_dev_dense_patterns", {})
        out = []
        for k, p in enumerate(factors):
            idx = p._indices()
            key = (idx.data_ptr(), idx.shape[1], str(idx.device))
            pat = cache.get(k)
            if pat is None or pat["key"] != key:
                pat = _dense_pattern(p)
                cache[k] = pat
            out.append(pat)
        return out

    def use_dense_path(self, batch: int) -> bool:
        """The batch-independent product of the factors is multiplied out (dense-product path) when the batch is large enough to
        amortise it; the sparse chain kernel (intermediates in shared memory) serves small batches and very wide factors.
        SNB200_PSM_PATH=dense|sparse forces a path."""
        import os
        forced = os.environ.get("SNB200_PSM_PATH", "")
        eligible = self._dense_eligible()
        if forced == "dense":
            assert eligible, "PSMLayer: the dense-product path needs output_dim % 4 == 0 and factor dimensions <= 16384"
            return True
        if forced == "sparse":
            return False
        return eligible and batch >= 1024

    def _dense_eligible(self) -> bool:
        return self.output_dim % 4 == 0 and max(max(p.shape) for p in self.sparse_matrices) <= 16384

    def use_dense_bf16_path(self) -> bool:
        """bfloat16 features take the dense-product path on bf16 tensor cores whenever the layer is eligible for it and
        SNB200_PSM_PATH does not force the sparse chain -- at every batch size, so the output dtype does not depend on the batch."""
        import os
        return os.environ.get("SNB200_PSM_PATH", "") != "sparse" and self._dense_eligible()

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop("_dev_patterns", None)
        state.pop("_dev_dense_patterns", None)
        state.pop("_dev_W_bf16", None)
        return state

    def forward(self, U):
        self._require_cuda(U, "PSMLayer.forward")
        assert U.dim() == 2 and U.shape[1] == self.input_dim, "PSMLayer expects a (batch, input_dim) input"
        bf16 = U.dtype == torch.bfloat16 and self.use_dense_bf16_path()    # bf16 output, float32 parameters and gradients
        if not bf16 and U.dtype != torch.float32:
            U = U.float()
        if not bf16 and U.stride(1) != 1:
            U = U.contiguous()
        # torch's sparse SGD update on CUDA (param.add_(sparse_grad)) concatenates the indices instead of summing
        # matching entries, so nnz grows with every step; fold duplicates back before using the pattern.
        for k, p in enumerate(self.sparse_matrices):
            if p._nnz() != self._base_nnz[k]:
                with torch.no_grad():
                    p.data = p.detach().coalesce()
                self._base_nnz[k] = int(p._nnz())
        if bf16:
            fn = _PSMDenseBF16Function
        else:
            fn = _PSMDenseFunction if self.use_dense_path(U.shape[0]) else _PSMFunction
        return fn.apply(U, self.bias if self.use_bias else None, self, *self.sparse_matrices)

    forward_sparse = forward   # the reference's alternative torch.sparse.mm path (psm_layer.py:36-45): same math

    def get_nb_parameters(self) -> int:
        return self.get_nb_parameters_in_weight_matrix() + len(self.bias)

    def get_nb_parameters_in_weight_matrix(self) -> int:
        return sum([len(mat.coalesce().values()) for mat in self.sparse_matrices])


def _factorize(weight: np.ndarray, nb_params_share: float):
    """The reference fits the factors with pyfaust's hierarchical PALM4MSA (approximators/psm_approximator.py:
    107-148), an unpinned PyPI dependency whose factorisation values no reference test pins (SURVEY.md
    section 8c) and which is out of scope here: a budget-respecting two-factor start: the largest-magnitude entries
    of W times a sparse identity -- enough for training from scratch; pass sparse_matrices=... for anything else."""
    out_dim, in_dim = weight.shape
    budget = int(nb_params_share * weight.size)
    mx = max(out_dim, in_dim)
    eye_nnz = min(in_dim, max(budget // 2, 0))
    keep = max(budget - eye_nnz, 0)
    W = np.zeros((out_dim, mx))
    W[:, :in_dim] = weight
    if keep < W.size:
        thresh = np.partition(np.abs(W).ravel(), W.size - keep)[W.size - keep] if keep > 0 else np.inf
        W = np.where(np.abs(W) >= thresh, W, 0.0)
        nz = np.flatnonzero(W)
        if len(nz) > keep:
            W.ravel()[nz[keep:]] = 0.0
    E = scipy.sparse.lil_matrix((mx, in_dim))
    for i in range(eye_nnz):
        E[i, i] = 1.0
    return [scipy.sparse.csr_matrix(W), scipy.sparse.csr_matrix(E)]


def build_PSMLayer_from_res_dict(res_dict: dict, bias: np.ndarray) -> PSMLayer:
    """reference layers/psm_layer.py:68-80 (the dense cross-check there needs a forward pass, i.e. a GPU here)."""
    sparse_matrices = res_dict["faust_approximation"]
    assert len(sparse_matrices) == res_dict["nb_matrices"], "Mismatch between expected and real number of matrices in the FAUST approximation"
    shape = res_dict["approx_mat_dense"].shape
    return PSMLayer(input_dim=shape[1], output_dim=shape[0], sparse_matrices=sparse_matrices, initial_bias=bias)
