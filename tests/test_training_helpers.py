"""Host logic of the training-loop mirror (reference training_helpers.py) with a plain CPU module, and the
reference's test_train_improvement on the CUDA layers (gpu)."""
import numpy as np
import pytest
import torch

from structurednets_b200 import training_helpers as TH


def toy(n=200, i=12, o=5, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1, 1, size=(n, i)).astype(np.float32)
    W = rng.uniform(-1, 1, size=(i, o)).astype(np.float32)
    return X, (X @ W).argmax(1).astype(np.int64)


def test_get_batch_slices_like_reference():
    X, y = toy()
    xb, yb = TH.get_batch(X, y, batch_size=64, batch_i=3)
    assert xb.shape == (8, 12) and yb.shape == (8,) and xb.dtype == torch.float32 and yb.dtype == torch.int64
    np.testing.assert_array_equal(xb.numpy(), X[192:200])
    xf, yf = TH.get_full_batch(X, y)
    assert xf.shape == (200, 12)


def test_train_contract_nine_tuple_and_early_stopping():
    torch.manual_seed(0)
    X, y = toy()
    model = torch.nn.Linear(12, 5)
    res = TH.train(model, X, y, patience=2, batch_size=50, lr=5e-2, min_patience_improvement=1e6, optimizer_class=torch.optim.SGD)
    assert len(res) == 9
    trained, s_tl, s_ta, s_vl, s_va, tlh, tah, vlh, vah = res
    assert isinstance(trained, torch.nn.Linear) and trained is not model          # restore_best_model -> pickled snapshot
    assert len(tlh) == len(vlh) == 3                                              # patience 2 + huge min improvement -> 3 epochs
    np.testing.assert_allclose(tlh, vlh)                                          # reference quirk: "val" history is the train set (:151)
    assert tlh[-1] < s_tl
    res2 = TH.train(model, X, y, patience=1, batch_size=50, lr=1e-2, restore_best_model=False, min_patience_improvement=1e6)
    assert res2[0] is model


def test_train_with_decreasing_lr_returns_lists_of_ten():
    X, y = toy(n=80)
    res = TH.train_with_decreasing_lr(torch.nn.Linear(12, 5), X, y, patience=1, batch_size=80, min_patience_improvement=1e6)
    assert len(res) == 9 and all(len(h) == 10 for h in res[1:])


def test_one_hot_targets_accuracy_path():
    X, y = toy()
    Y = np.eye(5, dtype=np.float32)[y]
    loss, acc = TH.get_loss_and_accuracy_for_model(torch.nn.Linear(12, 5), X, Y, loss_function_class=torch.nn.MSELoss, batch_size=64)
    assert 0.0 <= float(acc) <= 1.0 and float(loss) > 0


@pytest.mark.gpu
def test_train_improvement_all_layers(built_lib):
    """reference tests/test_layers.py:76-104: 20x20, share 0.5, MSE to ones, SGD lr 1e-3, full batch, through train()."""
    from structurednets_b200.layers.hmat_layer import HMatLayer
    from structurednets_b200.layers.ldr_layer import LDRLayer
    from structurednets_b200.layers.lr_layer import LRLayer
    from structurednets_b200.layers.psm_layer import PSMLayer
    from structurednets_b200.layers.sss_layer import SSSLayer
    from structurednets_b200.layers.tl_layer import TLLayer
    from structurednets_b200.synth import random_mixed_system
    np.random.seed(0)
    n = 1000
    X = np.random.uniform(-1, 1, size=(n, 20)).astype(np.float32)
    Y = np.ones((n, 20), dtype=np.float32)
    Xt = torch.tensor(X, device="cuda")
    layers = [LRLayer(20, 20, 0.5), PSMLayer(20, 20, nb_params_share=0.5), HMatLayer(20, 20, 0.5), LDRLayer(20, 20, 0.5), TLLayer(20, 20, 0.5),
              SSSLayer(20, 20, 0.5, nb_states=10, initial_system_approx=random_mixed_system(20, 20, 10, 2, seed=3))]
    for layer in layers:
        layer = layer.to("cuda")
        before = float((layer(Xt).detach() - 1).abs().max())
        trained, *_ = TH.train(model=layer, X_train=X, y_train=Y, patience=10, batch_size=n, verbose=False, lr=1e-3, restore_best_model=False,
                               loss_function_class=torch.nn.MSELoss, min_patience_improvement=1e6, optimizer_class=torch.optim.SGD, use_gpu=True)
        after = float((trained(Xt).detach() - 1).abs().max())
        assert after < before, type(layer).__name__ + " failed to improve the error"


def test_train_resident_matches_train_exactly_on_cpu():
    """Device-resident loop (SURVEY 8f rank 1): same RNG consumption, same batches, same float32 accumulation order -> the same
    9-tuple as the reference-shaped loop, bit for bit on a deterministic (CPU) module."""
    X, y = toy(n=230)
    Xv, yv = toy(n=50, seed=3)
    outs = []
    for fn in (TH.train, TH.train_resident):
        torch.manual_seed(1)
        np.random.seed(7)
        model = torch.nn.Linear(12, 5)
        outs.append(fn(model, X, y, X_val=Xv, y_val=yv, patience=2, batch_size=64, lr=5e-2, min_patience_improvement=1e-3,
                       optimizer_class=torch.optim.SGD))
    a, b = outs
    assert len(b) == 9 and len(a[5]) == len(b[5]) >= 3
    for i in range(1, 9):
        np.testing.assert_array_equal(np.asarray(a[i]), np.asarray(b[i]))
        assert np.asarray(a[i]).dtype == np.asarray(b[i]).dtype
    for pa, pb in zip(a[0].parameters(), b[0].parameters()):
        assert torch.equal(pa, pb)


def test_train_resident_one_hot_mse_targets():
    X, y = toy(n=120)
    Y = np.eye(5, dtype=np.float32)[y]
    np.random.seed(0)
    res = TH.train_resident(torch.nn.Linear(12, 5), X, Y, patience=1, batch_size=50, lr=1e-2, loss_function_class=torch.nn.MSELoss,
                            min_patience_improvement=1e6, optimizer_class=torch.optim.SGD)
    assert len(res) == 9 and len(res[5]) == 2 and res[5][-1] < res[1]


@pytest.mark.gpu
def test_train_resident_on_the_cuda_layers_with_flat_sgd(built_lib):
    """train() vs train_resident() with the fused flat-buffer SGD on an SSS layer (3 501 parameter tensors -> one update kernel)."""
    from structurednets_b200.layers.sss_layer import SSSLayer
    from structurednets_b200.synth import random_mixed_system
    rng = np.random.default_rng(5)
    X = rng.uniform(-1, 1, size=(600, 128)).astype(np.float32)
    y = rng.integers(0, 24, size=600).astype(np.int64)
    hist = []
    for fn, flat, graph in ((TH.train, False, False), (TH.train_resident, True, False), (TH.train_resident, True, True)):
        np.random.seed(11)
        layer = SSSLayer(128, 24, 0.9, nb_states=12, initial_system_approx=random_mixed_system(128, 24, 12, 16, seed=11)).to("cuda")
        opt = TH.FlatSGD.for_model(layer) if flat else torch.optim.SGD
        extra = dict(cuda_graph=True) if graph else {}
        res = fn(layer, X, y, X_val=X[:100], y_val=y[:100], patience=1, batch_size=200, lr=1e-1, restore_best_model=False,
                 min_patience_improvement=1e6, optimizer_class=opt, use_gpu=True, **extra)
        hist.append(res)
    a = hist[0]
    for b in hist[1:]:     # eager resident loop, then the CUDA-graph replayed step: same losses as train()
        assert len(a[5]) == len(b[5]) == 2
        np.testing.assert_allclose(np.asarray(a[5], dtype=np.float64), np.asarray(b[5], dtype=np.float64), rtol=1e-5)
        np.testing.assert_allclose(np.asarray(a[1], dtype=np.float64), np.asarray(b[1], dtype=np.float64), rtol=1e-6)
        assert b[5][-1] < b[1]


def test_flat_sgd_equals_torch_sgd_on_the_flat_buffer():
    """FlatSGD (one update over the layer's flat parameter buffer) against torch.optim.SGD over the 3n+1 parameter views (host logic:
    no kernels run, the gradients are synthetic)."""
    from structurednets_b200.layers.sss_layer import SSSLayer
    from structurednets_b200.synth import random_mixed_system
    layers = [SSSLayer(64, 16, 0.9, nb_states=4, initial_bias=np.linspace(-1, 1, 16), initial_system_approx=random_mixed_system(64, 16, 4, 8, seed=2))
              for _ in range(2)]
    opts = [TH.FlatSGD.for_model(layers[0])(layers[0].parameters(), 0.25), torch.optim.SGD(layers[1].parameters(), lr=0.25)]
    g = torch.Generator().manual_seed(0)
    for layer, opt in zip(layers, opts):
        layer._ensure_flat()
        opt.zero_grad()
    noise = torch.randn(layers[0].flat_parameters().numel(), generator=g)
    for layer in layers:
        layer._prepare_grad_accumulation().copy_(noise)
    for opt in opts:
        opt.step()
    assert opts[0].loose is None
    assert torch.equal(layers[0].flat_parameters(), layers[1].flat_parameters())
    for a, b in zip(layers[0].parameters(), layers[1].parameters()):
        assert torch.equal(a, b)


@pytest.mark.parametrize("loop", ["train", "train_resident"])
@pytest.mark.parametrize("tag,opt,restore", [("sgd_best", torch.optim.SGD, True), ("adam_last", torch.optim.Adam, False)])
def test_train_equals_the_reference_train_bit_for_bit(loop, tag, opt, restore):
    """tests/golden/train_linear.npz holds what the REFERENCE's training_helpers.train (:107-181) returns on a seeded
    torch.nn.Linear (generated by tests/golden/make_golden.py from the unmodified reference): start losses / accuracies, the four
    per-epoch histories (so also the epoch at which early stopping fires) and the weights of the returned model.  This repo's
    train and train_resident must reproduce all of it exactly."""
    from tests import golden_io as GIO
    from tests.golden.make_golden import train_case
    z = GIO.load("train_linear")
    X, y, Xv, yv = train_case()
    torch.manual_seed(5)
    np.random.seed(11)
    model = torch.nn.Linear(12, 5)
    res = getattr(TH, loop)(model, X, y, X_val=Xv, y_val=yv, patience=3, batch_size=50, lr=5e-2, restore_best_model=restore,
                            min_patience_improvement=1e-3, optimizer_class=opt)
    np.testing.assert_array_equal(np.asarray([float(v) for v in res[1:5]]), z[tag + "_start"])
    for name, h in zip(("tl", "ta", "vl", "va"), res[5:9]):
        np.testing.assert_array_equal(np.asarray([float(v) for v in h]), z[tag + "_" + name], err_msg=name)
    np.testing.assert_array_equal(res[0].weight.detach().numpy(), z[tag + "_W"])
    np.testing.assert_array_equal(res[0].bias.detach().numpy(), z[tag + "_b"])


def test_live_reference_train_when_the_reference_tree_is_present():
    """Same comparison against the imported reference itself (build container only; skipped on the GPU box)."""
    from oracle.ref_import import load_reference, reference_available
    if not reference_available():
        pytest.skip("the reference project is not part of this repository (set SNB200_REFERENCE to a checkout of "
                    "MatthiasKi/structurednets); tests/golden/train_linear.npz holds its results")
    load_reference()
    from structurednets import training_helpers as RTH
    from tests.golden.make_golden import train_case
    X, y, Xv, yv = train_case()
    out = []
    for mod in (RTH, TH):
        torch.manual_seed(3)
        np.random.seed(4)
        res = mod.train(torch.nn.Linear(12, 5), X, y, X_val=Xv, y_val=yv, patience=2, batch_size=64, lr=1e-1, optimizer_class=torch.optim.SGD,
                        min_patience_improvement=1e-4)
        out.append(([float(v) for v in res[1:5]], [[float(v) for v in h] for h in res[5:9]], res[0].weight.detach().numpy()))
    assert out[0][0] == out[1][0] and out[0][1] == out[1][1]
    np.testing.assert_array_equal(out[0][2], out[1][2])


@pytest.mark.gpu
def test_fused_loss_kernels_match_torch(built_lib):
    """sn_ce_loss / sn_mse_loss (csrc/train.cu) through FusedLoss: loss value, gradient of the model output and the number of correct
    predictions against torch.nn.CrossEntropyLoss / MSELoss + argmax (reference training_helpers.py:10-29,57-73)."""
    g = torch.Generator(device="cuda").manual_seed(0)
    for B, C in ((256, 1000), (77, 10), (1000, 24)):
        logits = (torch.randn((B, C), device="cuda", generator=g) * 3).requires_grad_(True)
        target = torch.randint(0, C, (B,), device="cuda", generator=g)
        ref = torch.nn.CrossEntropyLoss()(logits, target)
        gref, = torch.autograd.grad(ref, logits)
        fused = TH.FusedLoss(torch.nn.CrossEntropyLoss, "cuda")
        loss = fused(logits, target)
        gf, = torch.autograd.grad(loss, logits)
        assert abs(float(loss) - float(ref)) < 1e-5 * abs(float(ref))
        assert float((gf - gref).abs().max()) < 1e-6 * float(gref.abs().max()) + 1e-9
        assert int(fused.correct) == int((logits.argmax(1) == target).sum())
        onehot = torch.nn.functional.one_hot(target, C).float()
        refm = torch.nn.MSELoss()(logits, onehot)
        gm, = torch.autograd.grad(refm, logits)
        fm = TH.FusedLoss(torch.nn.MSELoss, "cuda")
        lm = fm(logits, onehot)
        gfm, = torch.autograd.grad(lm, logits)
        assert abs(float(lm) - float(refm)) < 1e-5 * abs(float(refm))
        assert float((gfm - gm).abs().max()) < 1e-6 * float(gm.abs().max()) + 1e-12
        assert int(fm.correct) == int((logits.argmax(1) == target).sum())
    # accumulation over batches + reset, evaluation under no_grad
    fused = TH.FusedLoss(torch.nn.CrossEntropyLoss, "cuda")
    with torch.no_grad():
        a = fused(logits.detach()[:100], target[:100]); b = fused(logits.detach()[100:], target[100:])
    assert abs(float(fused.loss_sum) - float(a) - float(b)) < 1e-5
    fused.reset()
    assert float(fused.loss_sum) == 0.0 and int(fused.correct) == 0


@pytest.mark.gpu
def test_flat_adam_and_sgd_kernels_match_torch(built_lib):
    """FlatAdam / FlatSGD (sn_flat_adam / sn_flat_sgd over the layer's flat buffers) against torch.optim.Adam / SGD over the parameter
    views, ten steps of synthetic gradients; grad_scale folds the data-parallel 1 / world factor in."""
    from structurednets_b200.layers.lr_layer import LRLayer
    for cls, tcls, kw in ((TH.FlatAdam, torch.optim.Adam, {}), (TH.FlatSGD, torch.optim.SGD, {})):
        np.random.seed(1)
        la = LRLayer(96, 40, 0.5).to("cuda")
        np.random.seed(1)
        lb = LRLayer(96, 40, 0.5).to("cuda")
        oa = cls.for_model(la, grad_scale=0.5)(la.parameters(), 1e-2)
        ob = tcls(lb.parameters(), lr=1e-2)
        g = torch.Generator(device="cuda").manual_seed(3)
        for step in range(10):
            noise = torch.randn(la.flat_parameters().numel(), device="cuda", generator=g)
            la._prepare_grad_accumulation().copy_(noise)
            lb._prepare_grad_accumulation().copy_(noise * 0.5)
            oa.step(); ob.step()
        err = float((la.flat_parameters() - lb.flat_parameters()).abs().max())
        assert err < 2e-6, (cls.__name__, err)


@pytest.mark.gpu
def test_train_resident_with_fused_loss_and_flat_adam(built_lib):
    """The device-resident loop with the fused loss / accuracy kernel and the flat Adam kernel (optionally replayed from a CUDA graph)
    follows train() with torch's CrossEntropyLoss + Adam on the same layer to float32 rounding."""
    from structurednets_b200.layers.sss_layer import SSSLayer
    from structurednets_b200.synth import random_mixed_system
    rng = np.random.default_rng(6)
    X = rng.uniform(-1, 1, size=(600, 128)).astype(np.float32)
    y = rng.integers(0, 24, size=600).astype(np.int64)
    hist = []
    for fn, fused, graph in ((TH.train, False, False), (TH.train_resident, True, False), (TH.train_resident, True, True)):
        np.random.seed(12)
        layer = SSSLayer(128, 24, 0.9, nb_states=12, initial_system_approx=random_mixed_system(128, 24, 12, 16, seed=12)).to("cuda")
        opt = TH.FlatAdam.for_model(layer) if fused else torch.optim.Adam
        extra = dict(fused_loss=True, cuda_graph=graph) if fused else {}
        res = fn(layer, X, y, X_val=X[:100], y_val=y[:100], patience=2, batch_size=200, lr=1e-3, restore_best_model=False,
                 min_patience_improvement=1e6, optimizer_class=opt, use_gpu=True, **extra)
        hist.append(res)
    a = hist[0]
    for b in hist[1:]:
        assert len(a[5]) == len(b[5]) == 3
        np.testing.assert_allclose(np.asarray(a[5], dtype=np.float64), np.asarray(b[5], dtype=np.float64), rtol=2e-5)
        np.testing.assert_allclose(np.asarray(a[6], dtype=np.float64), np.asarray(b[6], dtype=np.float64), atol=1e-6)
        np.testing.assert_allclose(np.asarray(a[1], dtype=np.float64), np.asarray(b[1], dtype=np.float64), rtol=1e-6)
