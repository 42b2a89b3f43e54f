"""The reference's own C implementation of the SSS forward (speed_comparison/run.c, compiled unmodified into oracle/_ref/run) as a
second checker: it must accept the oracle's output (CPU) and the CUDA kernels' output through the C ABI (gpu), and reject a
perturbed one.  run.c's own tolerance: 1e-3 absolute (run.c:177,357)."""
import numpy as np
import pytest
import torch

from oracle import layers_cpu as O
from oracle import run_c
from structurednets_b200.layers.sss_layer import SSSLayer
from structurednets_b200.synth import random_mixed_system

CASES = [dict(i=76, o=14, n=7, d=5, ragged=True), dict(i=128, o=24, n=12, d=16, ragged=False), dict(i=320, o=64, n=40, d=16, ragged=False)]


def _binary_or_skip():
    if run_c.build_ref() is None:
        pytest.skip("oracle/_ref/run is not built: it is compiled from the reference project's speed_comparison/run.c, which is not "
                    "part of this repository (set SNB200_REFERENCE to a checkout of MatthiasKi/structurednets)")


def _layer(case, seed=3):
    sysm = random_mixed_system(case["i"], case["o"], case["n"], case["d"], seed=seed, ragged_state_dims=case["ragged"])
    rng = np.random.default_rng(seed)
    layer = SSSLayer(case["i"], case["o"], 0.9, initial_bias=rng.uniform(-1, 1, size=case["o"]), nb_states=case["n"], initial_system_approx=sysm)
    u = rng.uniform(-1, 1, size=(1, case["i"])).astype(np.float32)
    return layer, u


def _lists(layer):
    return [[p.detach().cpu().numpy() for p in getattr(layer, n)] for n in "ABCDEFG"]


@pytest.mark.parametrize("case", CASES)
def test_reference_c_program_accepts_the_oracle_forward(case):
    _binary_or_skip()
    layer, u = _layer(case)
    lists = [[p.detach() for p in getattr(layer, n)] for n in "ABCDEFG"]
    y = O.sss_forward(torch.tensor(u), *lists, layer.bias.detach(), layer.dims_in, layer.dims_out).numpy().reshape(-1)
    ok, out = run_c.run_reference_check(*_lists(layer), layer.bias.detach().numpy(), u, y)
    assert ok, out
    bad = y.copy()
    bad[len(bad) // 2] += 1e-2     # ten times run.c's tolerance: must be rejected
    ok2, out2 = run_c.run_reference_check(*_lists(layer), layer.bias.detach().numpy(), u, bad)
    assert not ok2 and "Checksum mismatch for the SSS layer" in out2


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["tc", "simt"])
@pytest.mark.parametrize("case", CASES[1:])
def test_reference_c_program_accepts_the_cuda_forward(case, path, built_lib, monkeypatch):
    _binary_or_skip()
    monkeypatch.setenv("SNB200_SSS_PATH", path)
    layer, u = _layer(case)
    params = _lists(layer)
    bias = layer.bias.detach().numpy().copy()
    layer = layer.to("cuda")
    rng = np.random.default_rng(9)
    X = rng.uniform(-1, 1, size=(40, case["i"])).astype(np.float32)
    X[17] = u[0]                                           # the checked vector sits inside a batch
    y = layer(torch.tensor(X, device="cuda")).detach().cpu().numpy()[17]
    ok, out = run_c.run_reference_check(*params, bias, u, y)
    assert ok, out


def test_layer_description_round_trip_through_the_parser(tmp_path):
    """structurednets_b200.speed_comparison.run reads what prepare_run.py writes (same text format as oracle/run_c.py emits)."""
    from structurednets_b200.speed_comparison.run import parse_layer_description, sss_layer_from_description
    layer, u = _layer(CASES[0])
    lists = _lists(layer)
    y = np.arange(CASES[0]["o"], dtype=np.float32)
    p = str(tmp_path / "layer_description.txt")
    run_c.write_layer_description(p, *lists, layer.bias.detach().numpy(), u, y)
    d = parse_layer_description(p)
    assert d["input_size"] == 76 and d["output_size"] == 14 and d["nb_states"] == 7
    np.testing.assert_allclose(d["checksum_inp"].reshape(-1), u.reshape(-1), rtol=1e-7)
    np.testing.assert_allclose(d["sss_checksum_out"].reshape(-1), y)
    rebuilt = sss_layer_from_description(d)
    for name, mats in zip("ABCDEFG", lists):
        for a, b in zip(getattr(rebuilt, name), mats):
            np.testing.assert_allclose(a.detach().numpy(), b, rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(rebuilt.bias.detach().numpy(), layer.bias.detach().numpy(), rtol=1e-6)


@pytest.mark.gpu
def test_batched_run_tool_checks_like_run_c(tmp_path, built_lib, capsys):
    """The B200 counterpart of run.c: same file, same checksum protocol, batches 1 and 300; a wrong checksum fails with run.c's message."""
    from structurednets_b200.speed_comparison.run import run
    layer, u = _layer(CASES[2])
    lists = [[p.detach() for p in getattr(layer, n)] for n in "ABCDEFG"]
    y = O.sss_forward(torch.tensor(u), *lists, layer.bias.detach(), layer.dims_in, layer.dims_out).numpy().reshape(-1)
    p = str(tmp_path / "layer_description.txt")
    rng = np.random.default_rng(1)
    W = rng.uniform(-1, 1, size=(CASES[2]["o"], CASES[2]["i"])).astype(np.float32)
    run_c.write_layer_description(p, *_lists(layer), layer.bias.detach().numpy(), u, y, W=W, standard_bias=np.ones(CASES[2]["o"], dtype=np.float32))
    assert run(p, batches=(1, 300), iterations=3) == 0
    out = capsys.readouterr().out
    assert out.count("dense_time:") == 2 and out.count("sss_time:") == 2 and "ERROR" not in out
    y[5] += 0.01
    run_c.write_layer_description(p, *_lists(layer), layer.bias.detach().numpy(), u, y, W=W, standard_bias=np.ones(CASES[2]["o"], dtype=np.float32))
    assert run(p, batches=(1,), iterations=1) == 1
    assert "ERROR: Checksum mismatch for the SSS layer in dimension 5" in capsys.readouterr().out
