"""bf16 features on the dense-product layers (PSM dense path, H-matrix dense-block path, LDR, TL) against the float32 oracle --
needs a B200.  Stated bf16 tolerance, as for the low-rank bf16 path: 2e-2 relative to the largest entry of the compared tensor
(bf16 features, W and grad_y in the products, fp32 accumulation), the oracle evaluated on the bf16-rounded x and grad_y."""
import numpy as np
import pytest
import scipy.sparse
import torch

from oracle import layers_cpu as O
from structurednets_b200.hmatrix import HMatrix, build_hmat_block_cluster_tree
from structurednets_b200.layers.hmat_layer import HMatLayer
from structurednets_b200.layers.ldr_layer import LDRLayer
from structurednets_b200.layers.psm_layer import PSMLayer
from structurednets_b200.layers.tl_layer import TLLayer
from tests import golden_io as GIO

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 2e-2


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30)) if b.size else 0.0


def dense(g):
    return (g.to_dense() if g.is_sparse else g).detach().cpu().numpy()


def inputs(B, n_in, n_out, seed):
    """bf16-rounded features and output gradients (what the kernels see), as float32 CPU tensors."""
    rng = np.random.default_rng(seed)
    X = torch.tensor(rng.uniform(-1, 1, size=(B, n_in)).astype(np.float32)).bfloat16().float()
    gy = torch.tensor(rng.uniform(-1, 1, size=(B, n_out)).astype(np.float32) / B).bfloat16().float()
    return X, gy


def run_bf16(layer, X, gy):
    """bf16 fwd + bwd with grad_y = gy and an input that takes a gradient; returns (y, grad_x)."""
    x = X.to(DEV).bfloat16().requires_grad_(True)
    y = layer(x)
    assert y.dtype == torch.bfloat16 and y.shape == (X.shape[0], gy.shape[1])
    y.backward(gy.to(DEV).bfloat16())
    assert x.grad.dtype == torch.bfloat16 and x.grad.shape == X.shape
    return y.detach().float().cpu().numpy(), x.grad.float().cpu().numpy()


def oracle(fn, X, gy):
    Xo = X.clone().requires_grad_(True)
    yo = fn(Xo)
    (yo * gy).sum().backward()
    return yo.detach().numpy(), Xo.grad.numpy()


# ---------------------------------------------------------------- fixtures: layers with their oracle
def psm_case(i, o, S, seed=0):
    layer = PSMLayer(i, o, sparse_matrices=S)
    dense_f = [torch.tensor(s.toarray()).float().requires_grad_(True) for s in S]
    b = layer.bias.detach().clone().requires_grad_(True)
    return layer, lambda X: O.psm_forward(X, dense_f, b), dense_f, b


def psm_three_factors():
    i, o = 90, 44          # neither a multiple of 8: staged features, padded outputs
    mx = 96
    S = [scipy.sparse.random(o, mx, density=0.1, random_state=1, format="csr"), scipy.sparse.random(mx, mx, density=0.1, random_state=2, format="csr"),
         scipy.sparse.random(mx, i, density=0.1, random_state=3, format="csr")]
    return i, o, S


def psm_c3():
    from bench import PSMWorkload
    wl = PSMWorkload()
    return wl.input_dim, wl.output_dim, wl.factors()


def check_psm(i, o, S, B, seed):
    layer, fn, dense_f, b = psm_case(i, o, S)
    X, gy = inputs(B, i, o, seed)
    yo, gxo = oracle(fn, X, gy)
    layer = layer.to(DEV)
    y, gx = run_bf16(layer, X, gy)
    assert rel_err(y, yo) < TOL and rel_err(gx, gxo) < TOL
    assert rel_err(dense(layer.bias.grad), b.grad.numpy()) < TOL
    for k, p in enumerate(layer.sparse_matrices):
        assert p.dtype == torch.float32 and p.grad.dtype == torch.float32
        assert p.grad.is_sparse and p.grad._nnz() == p._nnz()                 # sparse grads on the parameter's own pattern
        assert rel_err(dense(p.grad), dense_f[k].grad.numpy() * (S[k].toarray() != 0)) < TOL


def test_psm_bf16_three_factors_unaligned(built_lib):
    check_psm(*psm_three_factors(), B=37, seed=11)


def test_psm_bf16_c3_shape(built_lib):
    check_psm(*psm_c3(), B=1024, seed=12)


def hmat_fixture_layer():
    z = GIO.load("hmat_40x64")
    tree = build_hmat_block_cluster_tree((40, 64), eta=0.5, min_block_size=2)
    leaves = {(l.row_range.start, l.row_range.stop, l.col_range.start, l.col_range.stop): l for l in tree.get_all_leaf_elements()}
    for (r0, r1, c0, c1, L, R) in GIO.hmat_components(z):
        leaves[(r0, r1, c0, c1)].set_hmatrix_component(L, R)
    return HMatLayer(64, 40, 0.9, initial_bias=z["bias"], initial_hmatrix=HMatrix(tree, shape=(40, 64)))


def hmat_c4h_layer():
    from bench import HMatWorkload
    np.random.seed(4000)
    return HMatLayer(2048, 1000, 0.2, initial_hmatrix=HMatWorkload().hmatrix())


@pytest.mark.parametrize("make,B", [(hmat_fixture_layer, 29), (hmat_c4h_layer, 1024)])
def test_hmat_bf16_vs_oracle(built_lib, make, B):
    layer = make()
    comps = [(c.row_range.start, c.row_range.stop, c.col_range.start, c.col_range.stop, c.left_lr.detach().clone().requires_grad_(True),
              c.right_lr.detach().clone().requires_grad_(True)) for c in layer.hmatrix_components]
    b = layer.bias.detach().clone().requires_grad_(True)
    X, gy = inputs(B, layer.input_dim, layer.output_dim, 40 + B)
    yo, gxo = oracle(lambda X: O.hmat_forward(X, comps, b, layer.output_dim), X, gy)
    layer = layer.to(DEV)
    assert layer._use_dense_path()
    y, gx = run_bf16(layer, X, gy)
    assert rel_err(y, yo) < TOL and rel_err(gx, gxo) < TOL
    assert rel_err(dense(layer.bias.grad), b.grad.numpy()) < TOL
    gl = np.concatenate([dense(c.left_lr.grad).ravel() for c in layer.hmatrix_components]); gl_o = np.concatenate([c[4].grad.numpy().ravel() for c in comps])
    gr = np.concatenate([dense(c.right_lr.grad).ravel() for c in layer.hmatrix_components]); gr_o = np.concatenate([c[5].grad.numpy().ravel() for c in comps])
    assert rel_err(gl, gl_o) < TOL and rel_err(gr, gr_o) < TOL
    flat_grad = layer.flat_grad()
    assert flat_grad.dtype == torch.float32 and layer.bias.grad.data_ptr() == flat_grad.data_ptr()   # grads stay views of the flat buffer


def ldr_fixture_layer():
    z = GIO.load("ldr_12")
    return LDRLayer(12, 12, 0.95, initial_bias=z["bias"], initial_representation_matrices=GIO.ldr_rep(z))


def ldr_512_layer():
    np.random.seed(22)
    layer = LDRLayer(512, 512, 0.098)
    assert layer.representation_matrices[2].shape == (512, 22)
    return layer


@pytest.mark.parametrize("make,B", [(ldr_fixture_layer, 19), (ldr_512_layer, 1024)])
def test_ldr_bf16_vs_oracle(built_lib, make, B):
    layer = make()
    n = layer.input_dim
    rep = [p.detach().clone().requires_grad_(True) for p in layer.representation_matrices]
    b = layer.bias.detach().clone().requires_grad_(True)
    X, gy = inputs(B, n, n, 60 + B)
    yo, gxo = oracle(lambda X: O.ldr_forward(X, rep, b, (n, n)), X, gy)
    layer = layer.to(DEV)
    y, gx = run_bf16(layer, X, gy)
    assert rel_err(y, yo) < TOL and rel_err(gx, gxo) < TOL
    assert rel_err(dense(layer.bias.grad), b.grad.numpy()) < TOL and layer.bias.grad.dtype == torch.float32
    A, Bm, G, H = layer.representation_matrices
    assert A.dtype == torch.float64 and A.is_sparse and A.grad.is_sparse and A.grad.dtype == torch.float64
    assert G.grad.dtype == torch.float64 and not G.grad.is_sparse
    for k, p in enumerate((A, Bm)):
        mask = rep[k].detach().to_dense().numpy() != 0
        assert rel_err(dense(p.grad), dense(rep[k].grad) * mask) < TOL
    assert rel_err(dense(G.grad), rep[2].grad.numpy()) < TOL and rel_err(dense(H.grad), rep[3].grad.numpy()) < TOL


def test_tl_bf16_vs_oracle(built_lib):
    z = GIO.load("tl_16")
    layer = TLLayer(16, 16, 0.5, initial_bias=z["bias"], initial_lr_matrices=[z["G"], z["H"]])
    Gt, Ht, b = [t.detach().clone().requires_grad_(True) for t in (layer.G, layer.H, layer.bias)]
    X, gy = inputs(23, 16, 16, 16)
    yo, gxo = oracle(lambda X: O.tl_forward(X, Gt, Ht, b), X, gy)
    layer = layer.to(DEV)
    y, gx = run_bf16(layer, X, gy)
    assert rel_err(y, yo) < TOL and rel_err(gx, gxo) < TOL
    assert rel_err(dense(layer.G.grad), Gt.grad.numpy()) < TOL and rel_err(dense(layer.H.grad), Ht.grad.numpy()) < TOL
    assert rel_err(dense(layer.bias.grad), b.grad.numpy()) < TOL
    assert layer.G.dtype == torch.float32 and layer.G.grad.dtype == torch.float32


# ---------------------------------------------------------------- parameter updates, fallbacks, graphs
def test_parameter_updates_reach_the_bf16_path(built_lib):
    """W is rebuilt from the current parameters on every bf16 call; fp32 calls on the same layer are unaffected."""
    np.random.seed(9)
    rng = np.random.default_rng(9)
    i, o, S = psm_three_factors()
    layers = [PSMLayer(i, o, sparse_matrices=S), hmat_fixture_layer(), ldr_fixture_layer(),
              TLLayer(16, 16, 0.5, initial_lr_matrices=[rng.uniform(-1, 1, (16, 4)) / 4, rng.uniform(-1, 1, (4, 16)) / 4])]
    for layer in layers:
        layer = layer.to(DEV)
        x = (torch.rand(64, layer.input_dim, device=DEV) * 2 - 1).bfloat16().float()
        y32 = layer(x)
        y16 = layer(x.bfloat16())
        assert y16.dtype == torch.bfloat16 and rel_err(y16.detach().float().cpu(), y32.detach().cpu()) < TOL
        with torch.no_grad():
            for p in layer.parameters():
                if p.is_sparse and isinstance(layer, PSMLayer):
                    p._values().mul_(1.5)
                elif not p.is_sparse and p.dim() == 2:        # (LDR: G and H only, A and B set how many powers matter)
                    p.mul_(1.5)
        y16b = layer(x.bfloat16())
        y32b = layer(x)
        assert rel_err(y16b.detach().float().cpu(), y32b.detach().cpu()) < TOL
        assert rel_err(y32b.detach().cpu(), y32.detach().cpu()) > 0.1      # the update changed the output


def test_fallbacks_keep_float32_output(built_lib, monkeypatch):
    """Paths without a bf16 variant upcast and return float32, exactly what the float32 input gives."""
    X, _ = inputs(37, 90, 44, 5)
    i, o, S = psm_three_factors()
    monkeypatch.setenv("SNB200_PSM_PATH", "sparse")
    layer = PSMLayer(i, o, sparse_matrices=S).to(DEV)
    y16, y32 = layer(X.to(DEV).bfloat16()), layer(X.to(DEV))
    assert y16.dtype == torch.float32 and rel_err(y16.detach().cpu(), y32.detach().cpu()) < 1e-6
    monkeypatch.delenv("SNB200_PSM_PATH")

    z = GIO.load("psm_50x30_2f")            # output_dim 30: not eligible for the dense-product path
    layer = PSMLayer(50, 30, initial_bias=z["bias"], sparse_matrices=[scipy.sparse.csr_matrix(z["f0_dense"]), scipy.sparse.csr_matrix(z["f1_dense"])]).to(DEV)
    xz = torch.tensor(z["X"], device=DEV).bfloat16()
    y16, y32 = layer(xz), layer(xz.float())
    assert y16.dtype == torch.float32 and rel_err(y16.detach().cpu(), y32.detach().cpu()) < 1e-6

    monkeypatch.setenv("SNB200_HMAT_PATH", "leaf")
    layer = hmat_fixture_layer().to(DEV)
    xh = (torch.rand(21, 64, device=DEV) * 2 - 1).bfloat16()
    y16, y32 = layer(xh), layer(xh.float())
    assert y16.dtype == torch.float32 and rel_err(y16.detach().cpu(), y32.detach().cpu()) < 1e-6


def test_psm_small_batch_bf16_takes_the_dense_path(built_lib):
    i, o, S = psm_three_factors()
    layer = PSMLayer(i, o, sparse_matrices=S).to(DEV)
    assert not layer.use_dense_path(64)
    y = layer((torch.rand(64, i, device=DEV) * 2 - 1).bfloat16())
    assert y.dtype == torch.bfloat16


@pytest.mark.parametrize("kind", ["psm", "hmat"])
def test_bf16_step_replays_in_a_cuda_graph(built_lib, kind):
    if kind == "psm":
        i, o, S = psm_three_factors()
        layer = PSMLayer(i, o, sparse_matrices=S).to(DEV)
    else:
        layer = hmat_c4h_layer().to(DEV)
    B = 512
    X, gy = inputs(B, layer.input_dim, layer.output_dim, 77)
    x = X.to(DEV).bfloat16().requires_grad_(True)
    g = gy.to(DEV).bfloat16()
    params = [p for p in layer.parameters()]

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
    for p in params:           # the captured backward binds fresh gradients (H-matrix: clears and rebinds its flat buffer)
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
