"""Empty batches through every layer path and dtype -- needs a B200.

An empty batch is a normal input: `distributed.shard_bounds` hands a rank an empty shard whenever the batch has fewer samples than
there are ranks, and slicing gives one too.  Each path gets `torch.empty(0, in)`, a leaf, and the empty slice `x[5:5]` of a real
tensor, a view that passes its gradient on to that tensor.  (torch reports data_ptr() == 0 for both; that the C entries neither read
nor check batch pointers when B = 0 is tested with dangling pointers in tests/test_empty_batch_abi.py.)  The forward must return a
(0, out) tensor of the dtype the DESIGN section 4.7 rule gives, the backward a (0, in) `grad_x`; parameter and bias gradients are
zero, as autograd's on an empty batch, and gradients already accumulated stay exactly as they were.
"""
import numpy as np
import pytest
import scipy.sparse
import torch

from structurednets_b200.layers.hmat_layer import HMatLayer
from structurednets_b200.layers.ldr_layer import LDRLayer
from structurednets_b200.layers.lr_layer import LRLayer
from structurednets_b200.layers.psm_layer import PSMLayer
from structurednets_b200.layers.sss_layer import SSSLayer
from structurednets_b200.layers.tl_layer import TLLayer
from structurednets_b200.synth import random_mixed_system

pytestmark = pytest.mark.gpu
DEV = "cuda"
F32, BF16 = torch.float32, torch.bfloat16


def sss():
    return SSSLayer(128, 24, 0.9, nb_states=12, initial_system_approx=random_mixed_system(128, 24, 12, 16, seed=11))


def psm():
    S = [scipy.sparse.random(44, 96, density=0.1, random_state=1, format="csr"), scipy.sparse.random(96, 96, density=0.1, random_state=2, format="csr"),
         scipy.sparse.random(96, 88, density=0.1, random_state=3, format="csr")]
    return PSMLayer(88, 44, sparse_matrices=S)


def hmat():
    np.random.seed(31)
    return HMatLayer(96, 72, 0.4)


# (layer, environment that selects the path, feature dtype, output dtype)
PATHS = {
    "sss_tc": (sss, {"SNB200_SSS_PATH": "tc"}, F32, F32),
    "sss_simt": (sss, {"SNB200_SSS_PATH": "simt"}, F32, F32),
    "psm_sparse": (psm, {"SNB200_PSM_PATH": "sparse"}, F32, F32),
    "psm_dense": (psm, {"SNB200_PSM_PATH": "dense"}, F32, F32),
    "psm_bf16": (psm, {}, BF16, BF16),
    "hmat_dense": (hmat, {"SNB200_HMAT_PATH": "dense"}, F32, F32),
    "hmat_leaf": (hmat, {"SNB200_HMAT_PATH": "leaf"}, F32, F32),
    "hmat_bf16": (hmat, {"SNB200_HMAT_PATH": "dense"}, BF16, BF16),
    "lr_f32": (lambda: LRLayer(256, 72, 0.57), {}, F32, F32),
    "lr_bf16": (lambda: LRLayer(256, 72, 0.57), {}, BF16, BF16),
    "ldr_f32": (lambda: LDRLayer(64, 64, 0.3), {}, F32, F32),
    "ldr_bf16": (lambda: LDRLayer(64, 64, 0.3), {}, BF16, BF16),
    "tl_f32": (lambda: TLLayer(16, 16, 0.5), {}, F32, F32),
    "tl_bf16": (lambda: TLLayer(16, 16, 0.5), {}, BF16, BF16),
}


def grads(layer):
    """name -> dense copy of .grad (None when unset) for every parameter that takes a gradient."""
    out = {}
    for n, p in layer.named_parameters():
        if p.requires_grad:
            g = p.grad
            out[n] = None if g is None else (g.to_dense() if g.is_sparse else g).detach().clone()
    return out


def empty_inputs(n_in, dtype):
    """torch.empty(0, n_in) and the empty slice [5:5] of a real (8, n_in) tensor, both taking a gradient."""
    a = torch.empty(0, n_in, device=DEV, dtype=dtype, requires_grad=True)
    full = torch.randn(8, n_in, device=DEV).to(dtype).requires_grad_(True)
    b = full[5:5]
    b.retain_grad()
    return [("empty", a), ("slice", b)]


def run(layer, x, out_dim, out_dtype):
    y = layer(x)
    assert y.shape == (x.shape[0], out_dim) and y.dtype == out_dtype
    y.float().sum().backward()
    return y


@pytest.mark.parametrize("path", sorted(PATHS))
def test_empty_batch_forward_and_backward(built_lib, monkeypatch, path):
    make, env, dtype, out_dtype = PATHS[path]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    torch.manual_seed(0)
    layer = make().to(DEV)
    n_in = layer.input_dim
    n_out = layer.output_dim

    # a fresh layer: an empty batch yields zero gradients, like autograd on an empty batch
    for what, x in empty_inputs(n_in, dtype):
        layer.zero_grad(set_to_none=True)
        run(layer, x, n_out, out_dtype)
        assert x.grad is not None and x.grad.shape == (0, n_in), (what, None if x.grad is None else x.grad.shape)
        for n, g in grads(layer).items():
            assert g is not None, (what, n)
            assert not bool(g.any()), (what, n)

    # gradients accumulated by a real batch stay exactly as they are
    layer.zero_grad(set_to_none=True)
    run(layer, torch.randn(8, n_in, device=DEV).to(dtype), n_out, out_dtype)
    before = grads(layer)
    assert all(g is not None for g in before.values())
    for what, x in empty_inputs(n_in, dtype):
        run(layer, x, n_out, out_dtype)
        assert x.grad.shape == (0, n_in)
        after = grads(layer)
        for n in before:
            assert torch.equal(after[n], before[n]), (what, n)
