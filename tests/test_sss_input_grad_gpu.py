"""Input gradients of SSSLayer on the SIMT path, and layers with frozen parameters on both paths -- needs a B200.

Tolerance as everywhere in the suite: max-abs error / max-abs of the compared tensor, 1e-5 in fp32.
"""
import numpy as np
import pytest
import torch

from oracle import layers_cpu as O
from structurednets_b200.layers.sss_layer import SSSLayer
from structurednets_b200.synth import random_mixed_system
from tests.test_sss_plan import CASES, oracle_lists

pytestmark = pytest.mark.gpu

RTOL = 1e-5
DEV = "cuda"


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def make_layer(i, o, n, d, ragged=False, use_bias=True, seed=0, share=0.9):
    sysm = random_mixed_system(i, o, n, d, seed=seed, ragged_state_dims=ragged)
    rng = np.random.default_rng(seed + 1)
    bias = rng.uniform(-1, 1, size=(o,)) if use_bias else None
    return SSSLayer(i, o, share, use_bias=use_bias, initial_bias=bias, nb_states=n, initial_system_approx=sysm)


def c1_layer(seed=1001):
    """BASELINE config C1: 4096 -> 1000, 500 stages, state dimension 16."""
    layer = SSSLayer(4096, 1000, 0.105, nb_states=500, initial_system_approx=random_mixed_system(4096, 1000, 500, 16, seed=seed))
    assert layer.statespace_dim == 16
    return layer


def inputs(B, i, o, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1, 1, size=(B, i)).astype(np.float32), rng.uniform(-1, 1, size=(B, o)).astype(np.float32)


def oracle(layer, X, gy):
    """y, grad_x, per-list parameter gradients and the bias gradient from autograd through the CPU oracle (layer still on the CPU)."""
    lists = oracle_lists(layer)
    b = layer.bias.detach().clone().requires_grad_(True) if layer.use_bias else None
    x = torch.tensor(X, requires_grad=True)
    yo = O.sss_forward(x, *lists, b, layer.dims_in, layer.dims_out)
    (yo * torch.tensor(gy)).sum().backward()
    return yo.detach().numpy(), x.grad.numpy(), list_grads(lists), (b.grad.numpy() if b is not None else None)


def list_grads(lists):
    """Oracle gradients of the lists A..G, flattened per list (parameters autograd never reached count as zero)."""
    return [np.concatenate([(p.grad.numpy() if p.grad is not None else np.zeros(tuple(p.shape), np.float32)).reshape(-1) for p in l])
            for l in lists]


def layer_grads(layer):
    return [np.concatenate([p.grad.detach().cpu().numpy().reshape(-1) for p in getattr(layer, name)]) for name in "ABCDEFG"]


def check_params(layer, go, gbo):
    for name, got, want in zip("ABCDEFG", layer_grads(layer), go):
        if want.size:
            assert rel_err(got, want) < RTOL, "grad " + name
    if gbo is not None:
        assert rel_err(layer.bias.grad.cpu().numpy(), gbo) < RTOL


def check_against_oracle(layer, X, gy, ref):
    """Forward + backward with grad_x of the layer (already on the GPU), everything compared with `ref` = oracle(...)."""
    yo, gxo, go, gbo = ref
    x = torch.tensor(X, device=DEV).requires_grad_(True)
    y = layer(x)
    assert rel_err(y.detach().cpu().numpy(), yo) < RTOL
    y.backward(torch.tensor(gy, device=DEV))
    assert rel_err(x.grad.cpu().numpy(), gxo) < RTOL, "grad_x"
    check_params(layer, go, gbo)


# ------------------------------------------------------------------------------------------------ oracle parity, SIMT path
SIMT_ONLY = [c for c in CASES if make_layer(c["i"], c["o"], c["n"], c["d"], c["ragged"]).build_tc_host_plan() is None]
EXTRA = [
    dict(i=96, o=30, n=6, d=20, B=40, ragged=False),     # state dimension above 16
    dict(i=340, o=32, n=2, d=16, B=19, ragged=False),    # 170 inputs per stage (> 160)
    dict(i=90, o=33, n=9, d=18, B=70, ragged=True),      # ragged state dimensions above 16
]


def test_the_imported_cases_include_tensor_core_ineligible_shapes():
    assert len(SIMT_ONLY) >= 4


@pytest.mark.parametrize("case", SIMT_ONLY + EXTRA)
@pytest.mark.parametrize("use_bias", [True, False])
def test_simt_grad_x_matches_oracle(case, use_bias, built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_SSS_PATH", "simt")
    layer = make_layer(case["i"], case["o"], case["n"], case["d"], case["ragged"], use_bias=use_bias)
    X, gy = inputs(case["B"], case["i"], case["o"], 3)
    ref = oracle(layer, X, gy)
    check_against_oracle(layer.to(DEV), X, gy, ref)


@pytest.mark.parametrize("B", [1, 53])
def test_simt_grad_x_single_sample_and_ragged_tile(B, built_lib, monkeypatch):
    """B = 1 and a batch that is not a multiple of the 48-sample tile, on the specialised C1-like stage shape and a generic one."""
    monkeypatch.setenv("SNB200_SSS_PATH", "simt")
    for case in (CASES[4], EXTRA[0]):
        layer = make_layer(case["i"], case["o"], case["n"], case["d"], case["ragged"])
        X, gy = inputs(B, case["i"], case["o"], 5)
        ref = oracle(layer, X, gy)
        check_against_oracle(layer.to(DEV), X, gy, ref)


def test_simt_grad_x_of_a_column_slice(built_lib, monkeypatch):
    """The input is a column slice of a wider tensor (row stride > input_dim); its gradient lands in the right columns."""
    monkeypatch.setenv("SNB200_SSS_PATH", "simt")
    case = CASES[2]
    layer = make_layer(case["i"], case["o"], case["n"], case["d"], case["ragged"])
    X, gy = inputs(37, case["i"], case["o"], 9)
    ref = oracle(layer, X, gy)
    layer = layer.to(DEV)
    wide = torch.zeros(37, case["i"] + 13, device=DEV)
    wide[:, 5:5 + case["i"]] = torch.tensor(X, device=DEV)
    wide.requires_grad_(True)
    x = wide[:, 5:5 + case["i"]]
    assert x.stride(0) > case["i"] and x.stride(1) == 1
    y = layer(x)
    assert rel_err(y.detach().cpu().numpy(), ref[0]) < RTOL
    y.backward(torch.tensor(gy, device=DEV))
    g = wide.grad.cpu().numpy()
    assert rel_err(g[:, 5:5 + case["i"]], ref[1]) < RTOL
    assert not g[:, :5].any() and not g[:, 5 + case["i"]:].any()
    check_params(layer, ref[2], ref[3])


# ------------------------------------------------------------------------------------------------ config size: the two paths agree
def test_c1_grad_x_simt_and_tc_agree_and_match_oracle(built_lib, monkeypatch):
    layer = c1_layer()
    B = 300
    X, gy = inputs(B, 4096, 1000, 1001)
    gy /= B
    ref = oracle(layer, X, gy)
    layer = layer.to(DEV)
    gxs = {}
    for path in ("simt", "tc"):
        monkeypatch.setenv("SNB200_SSS_PATH", path)
        for p in layer.parameters():
            p.grad = None
        x = torch.tensor(X, device=DEV).requires_grad_(True)
        layer(x).backward(torch.tensor(gy, device=DEV))
        gxs[path] = x.grad.cpu().numpy()
        assert rel_err(gxs[path], ref[1]) < RTOL, path
    assert rel_err(gxs["simt"], gxs["tc"]) < RTOL


# ------------------------------------------------------------------------------------------------ grad_x costs nothing when not asked for
@pytest.mark.parametrize("shape", ["c1", "d20"])
def test_simt_parameter_gradients_do_not_depend_on_grad_x(shape, built_lib, monkeypatch):
    """Parameter and bias gradients do not change when the backward also returns grad_x.  They are summed with float atomics across
    CTAs, so two backwards agree to rounding, not bitwise (also without grad_x); grad_x itself is bitwise reproducible (below)."""
    monkeypatch.setenv("SNB200_SSS_PATH", "simt")
    layer = (c1_layer() if shape == "c1" else make_layer(96, 30, 6, 20)).to(DEV)
    X, gy = inputs(1000, layer.input_dim, layer.output_dim, 21)
    gyd = torch.tensor(gy, device=DEV)
    flats = []
    for want_x in (False, True):
        for p in layer.parameters():
            p.grad = None
        x = torch.tensor(X, device=DEV).requires_grad_(want_x)
        layer(x).backward(gyd)
        assert (x.grad is not None) == want_x
        flats.append(layer.flat_grad().clone())
    assert rel_err(flats[1].cpu().numpy(), flats[0].cpu().numpy()) < 1e-6


def test_simt_grad_x_is_bitwise_reproducible_at_full_batch(built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_SSS_PATH", "simt")
    layer = c1_layer(7).to(DEV)
    g = torch.Generator(device=DEV).manual_seed(0)
    B = 8192
    x = (torch.rand(B, 4096, device=DEV, generator=g) * 2 - 1).requires_grad_(True)
    gy = (torch.rand(B, 1000, device=DEV, generator=g) * 2 - 1) / B
    y = layer(x)
    y.backward(gy, retain_graph=True)
    g1 = x.grad.clone()
    x.grad = None
    y.backward(gy)
    assert torch.isfinite(g1).all() and float(g1.abs().max()) > 0
    assert torch.equal(x.grad, g1)


# ------------------------------------------------------------------------------------------------ inside a network
def test_two_simt_layers_with_relu_between_match_oracle(built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_SSS_PATH", "simt")
    l1 = make_layer(31, 20, 7, 5, ragged=True, seed=2)
    l2 = make_layer(20, 9, 4, 3, seed=4)
    assert l1.build_tc_host_plan() is None and l2.build_tc_host_plan() is None
    X, gy = inputs(45, 31, 9, 13)
    o1, o2 = oracle_lists(l1), oracle_lists(l2)
    b1 = l1.bias.detach().clone().requires_grad_(True)
    b2 = l2.bias.detach().clone().requires_grad_(True)
    x = torch.tensor(X, requires_grad=True)
    h = torch.relu(O.sss_forward(x, *o1, b1, l1.dims_in, l1.dims_out))
    yo = O.sss_forward(h, *o2, b2, l2.dims_in, l2.dims_out)
    (yo * torch.tensor(gy)).sum().backward()

    l1, l2 = l1.to(DEV), l2.to(DEV)
    xd = torch.tensor(X, device=DEV).requires_grad_(True)
    y = l2(torch.relu(l1(xd)))
    assert rel_err(y.detach().cpu().numpy(), yo.detach().numpy()) < RTOL
    y.backward(torch.tensor(gy, device=DEV))
    for layer, lists, b in ((l1, o1, b1), (l2, o2, b2)):
        check_params(layer, list_grads(lists), b.grad.numpy())
    assert rel_err(xd.grad.cpu().numpy(), x.grad.numpy()) < RTOL


# ------------------------------------------------------------------------------------------------ frozen parameters
@pytest.mark.parametrize("path", ["simt", "tc"])
def test_frozen_layer_returns_grad_x_and_no_parameter_gradients(path, built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_SSS_PATH", path)
    case = CASES[4]   # inside the tensor-core limits, so both paths can run it
    layer = make_layer(case["i"], case["o"], case["n"], case["d"], case["ragged"])
    X, gy = inputs(70, case["i"], case["o"], 17)
    ref = oracle(layer, X, gy)
    layer = layer.to(DEV).requires_grad_(False)
    x = torch.tensor(X, device=DEV).requires_grad_(True)
    y = layer(x)
    assert rel_err(y.detach().cpu().numpy(), ref[0]) < RTOL
    y.backward(torch.tensor(gy, device=DEV))
    assert rel_err(x.grad.cpu().numpy(), ref[1]) < RTOL
    assert all(p.grad is None for p in layer.parameters())
    assert layer.__dict__.get("_flat_grad") is None
    with torch.no_grad():
        y2 = layer(x)
    assert not y2.requires_grad and y2.grad_fn is None
    y3 = layer(x.detach())
    assert not y3.requires_grad and y3.grad_fn is None
    assert rel_err(y2.cpu().numpy(), ref[0]) < RTOL


@pytest.mark.parametrize("path", ["simt", "tc"])
def test_trainable_bias_of_an_otherwise_frozen_layer_gets_its_gradient(path, built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_SSS_PATH", path)
    case = CASES[4]
    layer = make_layer(case["i"], case["o"], case["n"], case["d"], case["ragged"])
    X, gy = inputs(33, case["i"], case["o"], 19)
    ref = oracle(layer, X, gy)
    layer = layer.to(DEV).requires_grad_(False)
    layer.bias.requires_grad_(True)
    layer(torch.tensor(X, device=DEV)).backward(torch.tensor(gy, device=DEV))
    assert rel_err(layer.bias.grad.cpu().numpy(), ref[3]) < RTOL
    assert all(p.grad is None for n, p in layer.named_parameters() if n != "bias")


# ------------------------------------------------------------------------------------------------ CUDA graph
def test_simt_step_with_grad_x_replays_in_a_cuda_graph(built_lib, monkeypatch):
    monkeypatch.setenv("SNB200_SSS_PATH", "simt")
    layer = make_layer(96, 30, 6, 20).to(DEV)
    X, gy = inputs(200, 96, 30, 23)
    x = torch.tensor(X, device=DEV).requires_grad_(True)
    g = torch.tensor(gy, device=DEV)
    params = list(layer.parameters())

    def step():
        for p in params:
            p.grad = None
        x.grad = None
        y = layer(x)
        y.backward(g)
        return y.detach()

    def snapshot(y):
        return [y.cpu().clone(), x.grad.cpu().clone(), layer.flat_grad().cpu().clone()]

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
    got = snapshot(y.detach())
    assert torch.equal(got[0], eager[0]) and torch.equal(got[1], eager[1])   # y and grad_x: bitwise
    assert rel_err(got[2].numpy(), eager[2].numpy()) < 1e-6                  # parameter gradients: float atomics
