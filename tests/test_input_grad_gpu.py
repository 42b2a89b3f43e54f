"""The gradient w.r.t. the input features on the PSM sparse chain, the H-matrix leaf kernels and the bf16 low-rank path, with and
without parameter gradients, against autograd through the CPU oracle -- needs a B200.  Tolerance: max-abs error over max-abs of the
compared tensor; 1e-5 for float32, 2e-2 for bf16 against the float32 oracle on the bf16-rounded inputs."""
import numpy as np
import pytest
import scipy.sparse
import torch

from oracle import layers_cpu as O
from structurednets_b200.layers.hmat_layer import HMatLayer
from structurednets_b200.layers.lr_layer import LRLayer
from structurednets_b200.layers.psm_layer import PSMLayer
from tests import golden_io as GIO
from tests.test_dense_bf16_gpu import hmat_c4h_layer, hmat_fixture_layer, psm_c3, psm_three_factors

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5
TOL_BF16 = 2e-2


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30)) if b.size else 0.0


def dense(g):
    return (g.to_dense() if g.is_sparse else g).detach().cpu().numpy()


def data(B, n_in, n_out, seed, pad=0):
    """X (B x n_in, as a column slice of a wider array when pad > 0) and grad_y, float32 CPU."""
    rng = np.random.default_rng(seed)
    Xw = rng.uniform(-1, 1, size=(B, n_in + pad)).astype(np.float32)
    gy = rng.uniform(-1, 1, size=(B, n_out)).astype(np.float32) / max(B, 1)
    return torch.tensor(Xw), torch.tensor(gy)


def on_device(Xw, n_in, pad):
    """The device features as the layer sees them: a column slice (row pitch n_in + pad) that takes a gradient."""
    xw = Xw.to(DEV).requires_grad_(True)
    return xw, (xw[:, pad // 2:pad // 2 + n_in] if pad else xw)


# ---------------------------------------------------------------- PSM sparse chain
def psm_factors(nf):
    i, o, S = psm_three_factors()
    mx = 96
    if nf == 3:
        return i, o, S
    if nf == 2:
        return i, o, [scipy.sparse.random(o, mx, density=0.1, random_state=4, format="csr"), scipy.sparse.random(mx, i, density=0.1, random_state=5, format="csr")]
    return i, o, [scipy.sparse.random(o, i, density=0.2, random_state=6, format="csr")]


def psm_golden():
    z = GIO.load("psm_50x30_2f")
    return 50, 30, [scipy.sparse.csr_matrix(z["f0_dense"]), scipy.sparse.csr_matrix(z["f1_dense"])]


def psm_oracle(S, bias, Xs, gy):
    """grad_x, factor gradients (masked to the pattern) and bias gradient by autograd through the oracle."""
    dense_f = [torch.tensor(s.toarray()).float().requires_grad_(True) for s in S]
    b = bias.detach().cpu().clone().requires_grad_(True) if bias is not None else None
    X = Xs.clone().requires_grad_(True)
    (O.psm_forward(X, dense_f, b) * gy).sum().backward()
    return X.grad.numpy(), [d.grad.numpy() * (s.toarray() != 0) for d, s in zip(dense_f, S)], (b.grad.numpy() if b is not None else None)


def psm_run(layer, x, gy):
    for p in layer.parameters():
        p.grad = None
    (layer(x) * gy.to(DEV)).sum().backward()


PSM_CASES = [  # (factors, B, bias, pad)
    ("1f", 37, True, 0), ("2f", 37, True, 0), ("3f", 37, True, 0), ("3f", 1, True, 0), ("3f", 64, False, 0), ("3f", 29, True, 6),
    ("1f", 1, False, 6), ("golden", 37, True, 0), ("golden", 1, False, 0), ("golden", 2050, True, 4),
]


@pytest.mark.parametrize("case,B,bias,pad", PSM_CASES)
def test_psm_sparse_chain_grad_x_vs_oracle(built_lib, monkeypatch, case, B, bias, pad):
    monkeypatch.setenv("SNB200_PSM_PATH", "sparse")
    i, o, S = psm_golden() if case == "golden" else psm_factors(int(case[0]))
    layer = PSMLayer(i, o, use_bias=bias, sparse_matrices=S)
    Xw, gy = data(B, i, o, 100 + B + pad, pad)
    Xs = Xw[:, pad // 2:pad // 2 + i]
    gxo, gfo, gbo = psm_oracle(S, layer.bias if bias else None, Xs, gy)
    layer = layer.to(DEV)
    xw, x = on_device(Xw, i, pad)
    assert x.stride(0) == i + pad
    psm_run(layer, x, gy)
    assert rel_err(xw.grad[:, pad // 2:pad // 2 + i].cpu(), gxo) < RTOL
    if pad:
        assert not xw.grad[:, :pad // 2].any() and not xw.grad[:, pad // 2 + i:].any()
    for p, g in zip(layer.sparse_matrices, gfo):
        assert p.grad.is_sparse and p.grad._nnz() == p._nnz() and rel_err(dense(p.grad), g) < RTOL
    if bias:
        assert rel_err(dense(layer.bias.grad), gbo) < RTOL


def test_psm_sparse_chain_grad_x_at_c3(built_lib, monkeypatch):
    i, o, S = psm_c3()
    layer = PSMLayer(i, o, sparse_matrices=S)
    B = 256
    assert not layer.use_dense_path(B)        # the default selection at the reference's training batch
    Xw, gy = data(B, i, o, 256)
    gxo, gfo, gbo = psm_oracle(S, layer.bias, Xw, gy)
    layer = layer.to(DEV)
    x = Xw.to(DEV).requires_grad_(True)
    psm_run(layer, x, gy)
    assert rel_err(x.grad.cpu(), gxo) < RTOL and rel_err(dense(layer.bias.grad), gbo) < RTOL
    for p, g in zip(layer.sparse_matrices, gfo):
        assert rel_err(dense(p.grad), g) < RTOL


def test_psm_sparse_and_dense_grad_x_agree_at_c3(built_lib, monkeypatch):
    i, o, S = psm_c3()
    B = 1024
    Xw, gy = data(B, i, o, 1024)
    gx = {}
    for path in ("sparse", "dense"):
        monkeypatch.setenv("SNB200_PSM_PATH", path)
        layer = PSMLayer(i, o, sparse_matrices=S).to(DEV)
        x = Xw.to(DEV).requires_grad_(True)
        psm_run(layer, x, gy)
        gx[path] = x.grad.cpu()
    assert rel_err(gx["sparse"], gx["dense"]) < RTOL


@pytest.mark.parametrize("nf", [1, 3])
def test_psm_factor_gradients_unchanged_and_grad_x_bitwise_reproducible(built_lib, monkeypatch, nf):
    """nf = 1 runs the recomputing backward kernel, nf = 3 the one that reads the kept activations."""
    monkeypatch.setenv("SNB200_PSM_PATH", "sparse")
    i, o, S = psm_c3() if nf == 3 else psm_factors(1)
    layer = PSMLayer(i, o, sparse_matrices=S).to(DEV)
    Xw, gy = data(1024, i, o, 7)
    x0 = Xw.to(DEV)
    psm_run(layer, x0, gy)
    without = [dense(p.grad) for p in layer.sparse_matrices]
    gxs = []
    for _ in range(2):
        x = Xw.to(DEV).requires_grad_(True)
        psm_run(layer, x, gy)
        gxs.append(x.grad.cpu())
        for p, g in zip(layer.sparse_matrices, without):
            assert rel_err(dense(p.grad), g) < 1e-6     # float atomics across tiles: equal to rounding
    assert torch.equal(gxs[0], gxs[1])


def test_psm_bf16_features_on_the_sparse_chain_get_bf16_grad_x(built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_PSM_PATH", "sparse")
    i, o, S = psm_factors(3)
    layer = PSMLayer(i, o, sparse_matrices=S)
    Xw, gy = data(37, i, o, 5)
    Xb = Xw.bfloat16().float()
    gxo, _, _ = psm_oracle(S, layer.bias, Xb, gy)
    layer = layer.to(DEV)
    x = Xb.to(DEV).bfloat16().requires_grad_(True)
    y = layer(x)
    assert y.dtype == torch.float32
    (y * gy.to(DEV)).sum().backward()
    assert x.grad.dtype == torch.bfloat16 and rel_err(x.grad.float().cpu(), gxo) < TOL_BF16


def test_psm_grad_x_only_backward_leaves_the_forward_launchable(built_lib, monkeypatch):
    """The input-gradient-only backward launches the forward kernel with a small layer's shared memory; a larger layer's forward
    afterwards must still get the shared memory it needs."""
    monkeypatch.setenv("SNB200_PSM_PATH", "sparse")
    i, o, S = psm_c3()
    big = PSMLayer(i, o, sparse_matrices=S).to(DEV)
    xb = torch.rand(8, i, device=DEV)
    y0 = big(xb).detach()
    small_i, small_o, small_S = psm_factors(3)
    small = PSMLayer(small_i, small_o, sparse_matrices=small_S).to(DEV)
    freeze(small, False)
    x = torch.rand(8, small_i, device=DEV, requires_grad=True)
    small(x).sum().backward()
    assert x.grad is not None
    assert torch.equal(big(xb).detach(), y0)


# ---------------------------------------------------------------- H-matrix leaf kernels
def hmat_random_layer(bias=True):
    np.random.seed(31)
    return HMatLayer(96, 72, 0.4, use_bias=bias)


def hmat_fixture_no_bias():
    layer = hmat_fixture_layer()
    return HMatLayer(64, 40, 0.9, use_bias=False, initial_hmatrix=layer.hmatrix)


def hmat_oracle(layer, Xs, gy):
    comps = [(c.row_range.start, c.row_range.stop, c.col_range.start, c.col_range.stop, c.left_lr.detach().cpu().clone().requires_grad_(True),
              c.right_lr.detach().cpu().clone().requires_grad_(True)) for c in layer.hmatrix_components]
    b = layer.bias.detach().cpu().clone().requires_grad_(True) if layer.use_bias else None
    X = Xs.clone().requires_grad_(True)
    (O.hmat_forward(X, comps, b, layer.output_dim) * gy).sum().backward()
    gl = np.concatenate([c[4].grad.numpy().ravel() for c in comps])
    gr = np.concatenate([c[5].grad.numpy().ravel() for c in comps])
    return X.grad.numpy(), gl, gr, (b.grad.numpy() if b is not None else None)


def hmat_grads(layer):
    gl = np.concatenate([dense(c.left_lr.grad).ravel() for c in layer.hmatrix_components])
    gr = np.concatenate([dense(c.right_lr.grad).ravel() for c in layer.hmatrix_components])
    return gl, gr


@pytest.mark.parametrize("make,B,pad", [(hmat_fixture_layer, 1, 0), (hmat_fixture_layer, 13, 0), (hmat_fixture_no_bias, 29, 6),
                                        (hmat_random_layer, 1, 0), (hmat_random_layer, 37, 4), (lambda: hmat_random_layer(False), 19, 0)])
def test_hmat_leaf_grad_x_vs_oracle(built_lib, monkeypatch, make, B, pad):
    monkeypatch.setenv("SNB200_HMAT_PATH", "leaf")
    layer = make()
    i, o = layer.input_dim, layer.output_dim
    Xw, gy = data(B, i, o, 200 + B, pad)
    gxo, glo, gro, gbo = hmat_oracle(layer, Xw[:, pad // 2:pad // 2 + i], gy)
    layer = layer.to(DEV)
    assert not layer._use_dense_path()
    xw, x = on_device(Xw, i, pad)
    (layer(x) * gy.to(DEV)).sum().backward()
    assert rel_err(xw.grad[:, pad // 2:pad // 2 + i].cpu(), gxo) < RTOL
    gl, gr = hmat_grads(layer)
    assert rel_err(gl, glo) < 2 * RTOL and rel_err(gr, gro) < 2 * RTOL
    if layer.use_bias:
        assert rel_err(dense(layer.bias.grad), gbo) < RTOL


def test_hmat_leaf_and_dense_grad_x_agree_at_c4h(built_lib, monkeypatch):
    B = 8192
    gx = {}
    for path in ("leaf", "dense"):
        monkeypatch.setenv("SNB200_HMAT_PATH", path)
        layer = hmat_c4h_layer().to(DEV)
        Xw, gy = data(B, layer.input_dim, layer.output_dim, 8192)
        x = Xw.to(DEV).requires_grad_(True)
        (layer(x) * gy.to(DEV)).sum().backward()
        gx[path] = x.grad.cpu()
    assert rel_err(gx["leaf"], gx["dense"]) < RTOL


def test_hmat_default_selection_of_the_leaf_path_returns_grad_x(built_lib):
    layer = hmat_random_layer()
    layer.DENSE_PATH_MAX_ELEMENTS = 100          # this instance counts as too large to densify
    Xw, gy = data(45, layer.input_dim, layer.output_dim, 45)
    gxo, _, _, _ = hmat_oracle(layer, Xw, gy)
    layer = layer.to(DEV)
    assert not layer._use_dense_path()
    x = Xw.to(DEV).requires_grad_(True)
    (layer(x) * gy.to(DEV)).sum().backward()
    assert rel_err(x.grad.cpu(), gxo) < RTOL


# ---------------------------------------------------------------- bf16 low rank
def lr_rank72_layer():
    rng = np.random.default_rng(72)
    return LRLayer(256, 200, 0.5, initial_lr_components=[rng.uniform(-1, 1, (200, 72)) / 9, rng.uniform(-1, 1, (72, 256)) / 16])


def lr_oracle_bf16(layer, Xb, gyb):
    L, R = (t.detach().cpu().clone().requires_grad_(True) for t in (layer.left_lr, layer.right_lr))
    b = layer.bias.detach().cpu().clone().requires_grad_(True) if layer.use_bias else None
    X = Xb.clone().requires_grad_(True)
    (O.lr_forward(X, L, R, b) * gyb).sum().backward()
    return X.grad.numpy(), L.grad.numpy(), R.grad.numpy(), (b.grad.numpy() if b is not None else None)


def lr_run_bf16(layer, Xb, gyb):
    x = Xb.to(DEV).bfloat16().requires_grad_(True)
    y = layer(x)
    y.backward(gyb.to(DEV).bfloat16())
    assert x.grad.dtype == torch.bfloat16 and x.grad.shape == Xb.shape
    return x.grad


@pytest.mark.parametrize("make,B", [(lambda: LRLayer(2048, 1000, 0.1906), 512), (lambda: LRLayer(256, 72, 0.57), 300), (lambda: LRLayer(256, 72, 0.57), 1),
                                    (lr_rank72_layer, 300), (lr_rank72_layer, 37)])
def test_lr_bf16_grad_x_vs_oracle(built_lib, make, B):
    np.random.seed(7)
    layer = make()
    i, o = layer.input_dim, layer.output_dim
    Xw, gy = data(B, i, o, 300 + B)
    Xb, gyb = Xw.bfloat16().float(), gy.bfloat16().float()
    gxo, glo, gro, gbo = lr_oracle_bf16(layer, Xb, gyb)
    layer = layer.to(DEV)
    gx = lr_run_bf16(layer, Xb, gyb)
    assert rel_err(gx.float().cpu(), gxo) < TOL_BF16
    assert rel_err(dense(layer.left_lr.grad), glo) < TOL_BF16 and rel_err(dense(layer.right_lr.grad), gro) < TOL_BF16
    assert rel_err(dense(layer.bias.grad), gbo) < TOL_BF16


def test_lr_bf16_grad_x_bitwise_reproducible(built_lib):
    np.random.seed(8)
    layer = LRLayer(2048, 1000, 0.1906).to(DEV)
    Xw, gy = data(8192, 2048, 1000, 8)
    gxs = []
    for _ in range(2):
        layer.zero_grad(set_to_none=True)
        gxs.append(lr_run_bf16(layer, Xw, gy).cpu())
    assert torch.equal(gxs[0], gxs[1])


# ---------------------------------------------------------------- frozen parameters
def freeze(layer, keep_bias):
    for n, p in layer.named_parameters():
        p.requires_grad_(keep_bias and n == "bias")


@pytest.mark.parametrize("keep_bias", [False, True])
def test_frozen_psm_sparse_chain(built_lib, monkeypatch, keep_bias):
    monkeypatch.setenv("SNB200_PSM_PATH", "sparse")
    i, o, S = psm_factors(3)
    layer = PSMLayer(i, o, sparse_matrices=S)
    Xw, gy = data(37, i, o, 41)
    gxo, _, gbo = psm_oracle(S, layer.bias, Xw, gy)
    layer = layer.to(DEV)
    freeze(layer, keep_bias)
    x = Xw.to(DEV).requires_grad_(True)
    (layer(x) * gy.to(DEV)).sum().backward()
    assert rel_err(x.grad.cpu(), gxo) < RTOL
    assert all(p.grad is None for p in layer.sparse_matrices)
    assert (layer.bias.grad is not None and rel_err(dense(layer.bias.grad), gbo) < RTOL) if keep_bias else layer.bias.grad is None


@pytest.mark.parametrize("keep_bias", [False, True])
def test_frozen_hmat_leaf(built_lib, monkeypatch, keep_bias):
    monkeypatch.setenv("SNB200_HMAT_PATH", "leaf")
    layer = hmat_random_layer()
    Xw, gy = data(37, layer.input_dim, layer.output_dim, 42)
    gxo, _, _, gbo = hmat_oracle(layer, Xw, gy)
    layer = layer.to(DEV)
    freeze(layer, keep_bias)
    x = Xw.to(DEV).requires_grad_(True)
    (layer(x) * gy.to(DEV)).sum().backward()
    assert rel_err(x.grad.cpu(), gxo) < RTOL
    for c in layer.hmatrix_components:
        assert c.left_lr.grad is None and c.right_lr.grad is None
    if keep_bias:
        assert rel_err(dense(layer.bias.grad), gbo) < RTOL
    else:
        assert layer.bias.grad is None and layer.__dict__.get("_flat_grad") is None     # the flat gradient buffer is never allocated


@pytest.mark.parametrize("keep_bias", [False, True])
def test_frozen_lr_bf16(built_lib, keep_bias):
    np.random.seed(9)
    layer = LRLayer(256, 72, 0.57)
    Xw, gy = data(64, 256, 72, 43)
    Xb, gyb = Xw.bfloat16().float(), gy.bfloat16().float()
    gxo, _, _, gbo = lr_oracle_bf16(layer, Xb, gyb)
    layer = layer.to(DEV)
    freeze(layer, keep_bias)
    gx = lr_run_bf16(layer, Xb, gyb)
    assert rel_err(gx.float().cpu(), gxo) < TOL_BF16
    assert layer.left_lr.grad is None and layer.right_lr.grad is None
    if keep_bias:
        assert rel_err(dense(layer.bias.grad), gbo) < TOL_BF16
    else:
        assert layer.bias.grad is None and layer.__dict__.get("_flat_grad") is None


# ---------------------------------------------------------------- in a network
def psm_oracle_module(S, bias):
    dense_f = [torch.tensor(s.toarray()).float().requires_grad_(True) for s in S]
    b = bias.detach().cpu().clone().requires_grad_(True)
    return (lambda X: O.psm_forward(X, dense_f, b)), dense_f + [b], [s.toarray() != 0 for s in S] + [None]


def hmat_oracle_module(layer):
    comps = [(c.row_range.start, c.row_range.stop, c.col_range.start, c.col_range.stop, c.left_lr.detach().cpu().clone().requires_grad_(True),
              c.right_lr.detach().cpu().clone().requires_grad_(True)) for c in layer.hmatrix_components]
    b = layer.bias.detach().cpu().clone().requires_grad_(True)
    return (lambda X: O.hmat_forward(X, comps, b, layer.output_dim)), [b] + [t for c in comps for t in (c[4], c[5])]


def hmat_ref_grads(params):
    return [params[0].grad.numpy(), np.concatenate([t.grad.numpy().ravel() for t in params[1:]])]


def layer_grads(layer):
    if isinstance(layer, PSMLayer):
        return [dense(p.grad) for p in layer.sparse_matrices] + [dense(layer.bias.grad)]
    if isinstance(layer, HMatLayer):   # the leaf gradients compared as one tensor, as in tests/test_dense_bf16_gpu.py
        return [dense(layer.bias.grad), np.concatenate([dense(t.grad).ravel() for c in layer.hmatrix_components for t in (c.left_lr, c.right_lr)])]
    return [dense(layer.bias.grad), dense(layer.left_lr.grad), dense(layer.right_lr.grad)]


def test_psm_relu_psm_stack(built_lib):
    i, o, S1 = psm_factors(3)
    S2 = [scipy.sparse.random(24, o, density=0.2, random_state=8, format="csr"), scipy.sparse.random(o, o, density=0.2, random_state=9, format="csr")]
    first, second = PSMLayer(i, o, sparse_matrices=S1), PSMLayer(o, 24, sparse_matrices=S2)
    assert not first.use_dense_path(256)
    f, fp, fm = psm_oracle_module(S1, first.bias)
    s, sp, sm = psm_oracle_module(S2, second.bias)
    Xw, gy = data(256, i, 24, 500)
    X = Xw.clone().requires_grad_(True)
    (s(torch.relu(f(X))) * gy).sum().backward()
    first, second = first.to(DEV), second.to(DEV)
    x = Xw.to(DEV).requires_grad_(True)
    (second(torch.relu(first(x))) * gy.to(DEV)).sum().backward()
    assert rel_err(x.grad.cpu(), X.grad.numpy()) < RTOL
    for got, p, m in zip(layer_grads(first) + layer_grads(second), fp + sp, fm + sm):
        assert rel_err(got, p.grad.numpy() * (m if m is not None else 1)) < RTOL


def test_hmat_leaf_relu_psm_stack(built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_HMAT_PATH", "leaf")
    first = hmat_random_layer()
    S2 = [scipy.sparse.random(24, 72, density=0.2, random_state=10, format="csr"), scipy.sparse.random(72, 72, density=0.2, random_state=11, format="csr")]
    second = PSMLayer(72, 24, sparse_matrices=S2)
    f, fp = hmat_oracle_module(first)
    s, sp, sm = psm_oracle_module(S2, second.bias)
    Xw, gy = data(256, 96, 24, 501)
    X = Xw.clone().requires_grad_(True)
    (s(torch.relu(f(X))) * gy).sum().backward()
    first, second = first.to(DEV), second.to(DEV)
    x = Xw.to(DEV).requires_grad_(True)
    (second(torch.relu(first(x))) * gy.to(DEV)).sum().backward()
    assert rel_err(x.grad.cpu(), X.grad.numpy()) < RTOL
    for got, ref in zip(layer_grads(first), hmat_ref_grads(fp)):
        assert rel_err(got, ref) < 2 * RTOL
    for got, p, m in zip(layer_grads(second), sp, sm):
        assert rel_err(got, p.grad.numpy() * (m if m is not None else 1)) < RTOL


def test_bf16_hmat_dense_then_lr_stack(built_lib):
    first = hmat_random_layer()
    np.random.seed(12)
    second = LRLayer(72, 40, 0.63)
    assert second.left_lr.shape[1] == 16
    f, fp = hmat_oracle_module(first)
    L, R, b = (t.detach().clone().requires_grad_(True) for t in (second.left_lr, second.right_lr, second.bias))
    Xw, gy = data(256, 96, 40, 502)
    Xb, gyb = Xw.bfloat16().float(), gy.bfloat16().float()
    X = Xb.clone().requires_grad_(True)
    (O.lr_forward(f(X).bfloat16().float(), L, R, b) * gyb).sum().backward()
    first, second = first.to(DEV), second.to(DEV)
    assert first._use_dense_path()
    x = Xb.to(DEV).bfloat16().requires_grad_(True)
    h = first(x)
    assert h.dtype == torch.bfloat16
    y = second(h)
    y.backward(gyb.to(DEV).bfloat16())
    assert x.grad.dtype == torch.bfloat16 and rel_err(x.grad.float().cpu(), X.grad.numpy()) < TOL_BF16
    for got, ref in zip(layer_grads(first) + layer_grads(second), hmat_ref_grads(fp) + [t.grad.numpy() for t in (b, L, R)]):
        assert rel_err(got, ref) < TOL_BF16


# ---------------------------------------------------------------- CUDA graphs
@pytest.mark.parametrize("kind", ["psm", "hmat", "lr_bf16"])
def test_step_with_grad_x_replays_in_a_cuda_graph(built_lib, monkeypatch, kind):
    if kind == "psm":
        monkeypatch.setenv("SNB200_PSM_PATH", "sparse")
        i, o, S = psm_factors(3)
        layer = PSMLayer(i, o, sparse_matrices=S)
    elif kind == "hmat":
        monkeypatch.setenv("SNB200_HMAT_PATH", "leaf")
        layer = hmat_random_layer()
    else:
        np.random.seed(13)
        layer = LRLayer(256, 72, 0.57)
    layer = layer.to(DEV)
    Xw, gy = data(256, layer.input_dim, layer.output_dim, 600)
    bf16 = kind == "lr_bf16"
    x = (Xw.to(DEV).bfloat16() if bf16 else Xw.to(DEV)).requires_grad_(True)
    g = gy.to(DEV).bfloat16() if bf16 else gy.to(DEV)
    params = list(layer.parameters())

    def step():
        for p in params:
            p.grad = None
        x.grad = None
        y = layer(x)
        y.backward(g)
        return y.detach()

    def snapshot(y):
        return [y.float().cpu().numpy(), x.grad.float().cpu().numpy()] + [dense(p.grad) for p in params]

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            eager = snapshot(step())
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    for p in params:
        p.grad = None
    x.grad = None
    with torch.cuda.graph(graph):
        y = layer(x)
        y.backward(g)
    graph.replay()
    torch.cuda.synchronize()
    got = [y.detach().float().cpu().numpy(), x.grad.float().cpu().numpy()] + [dense(p.grad) for p in params]
    for a, b in zip(got, eager):
        assert rel_err(a, b) < 1e-5
