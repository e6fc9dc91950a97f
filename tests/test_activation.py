"""Dice (reference layers/activation.py:6-45) and the activation factory: pure torch modules, checked on CPU against the
formula and against what the reference module computed on the same inputs (tests/golden/dice.npz); the GPU test runs
the Dice tower (fused linears from libctr_b200.so + Dice between them) against the same computation in plain torch."""
import json
import os

import numpy as np
import pytest
import torch

from deepctr_torch_b200.layers import DNN, Dice, activation_layer
from helpers import GOLDEN_DIR


def _dice_golden():
    return np.load(os.path.join(GOLDEN_DIR, "dice.npz"), allow_pickle=False)


@pytest.mark.parametrize("dim,shape", [(2, (64, 8)), (3, (16, 5, 8))])
def test_dice_formula_and_reference(dim, shape):
    torch.manual_seed(0)
    d = Dice(shape[-1], dim)
    with torch.no_grad():
        d.alpha.copy_(torch.randn_like(d.alpha))
        d.bn.weight.copy_(torch.rand(shape[-1]) + 0.5)
        d.bn.bias.copy_(torch.randn(shape[-1]) * 0.1)
    x = torch.randn(*shape)
    d.train()
    flat = x.reshape(-1, shape[-1])
    mean, var = flat.mean(0), flat.var(0, unbiased=False)
    gate = torch.sigmoid((x - mean) / torch.sqrt(var + 1e-8) * d.bn.weight + d.bn.bias)
    alpha = d.alpha.reshape(-1)
    expect = gate * x + alpha * (1 - gate) * x
    assert torch.allclose(d(x), expect, atol=1e-6, rtol=1e-5)
    # the reference module from the same seeded state and inputs, train mode then eval mode (golden/make_golden.py)
    z, tag = _dice_golden(), "dim%d" % dim
    d = Dice(shape[-1], dim)
    d.load_state_dict({k[len(tag) + 7:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(tag + "/state/")})
    assert torch.equal(x, torch.from_numpy(z[tag + "/x"]))
    for mode, key in ((True, "/y_train"), (False, "/y_eval")):
        d.train(mode)
        ref = torch.from_numpy(z[tag + key])
        # the batch statistics are reductions whose rounding depends on the CPU and the thread count, so the stored
        # outputs match to round-off rather than bit for bit
        assert float((d(x) - ref).abs().max()) <= 1e-6 * float(ref.abs().max())


def test_dice_tower_keys_and_factory():
    tower = DNN(10, [8, 4], activation="dice", dice_dim=2)
    keys = list(tower.state_dict().keys())
    assert "activation_layers.0.alpha" in keys and "activation_layers.1.bn.running_var" in keys
    assert keys == json.loads(str(_dice_golden()["dnn_dice_keys"]))
    assert isinstance(activation_layer("dice", 8, 2), Dice)
    assert isinstance(activation_layer("prelu"), torch.nn.PReLU)
    with pytest.raises(NotImplementedError):
        activation_layer("swish")
    with pytest.raises(ValueError):          # the reference asserts on the same mismatch (dice_dim defaults to 3 in DNN)
        Dice(8, 3)(torch.randn(4, 8))


@pytest.mark.gpu
def test_dice_tower_on_gpu_matches_torch():
    torch.manual_seed(1)
    dev = "cuda:0"
    tower = DNN(24, [16, 8], activation="dice", dice_dim=2, init_std=0.1, device=dev)
    with torch.no_grad():
        for layer in tower.activation_layers:
            layer.alpha.copy_(torch.randn_like(layer.alpha) * 0.3)
    x = torch.randn(512, 24, device=dev, requires_grad=True)
    tower.train()
    y = tower(x)
    y.square().sum().backward()
    got = [x.grad.clone()] + [p.grad.clone() for p in tower.parameters()]
    # the same tower in plain torch (fp64), fresh batch-norm buffers
    x2 = x.detach().double().requires_grad_(True)
    params = [p.detach().double().requires_grad_(True) for p in tower.parameters()]
    named = dict(zip([k for k, _ in tower.named_parameters()], params))
    h = x2
    for i in range(2):
        z = torch.nn.functional.linear(h, named["linears.%d.weight" % i], named["linears.%d.bias" % i])
        gate = torch.sigmoid(torch.nn.functional.batch_norm(z, None, None, named["activation_layers.%d.bn.weight" % i],
                                                            named["activation_layers.%d.bn.bias" % i], training=True, eps=1e-8))
        h = gate * z + named["activation_layers.%d.alpha" % i] * (1 - gate) * z
    h.square().sum().backward()
    assert float((y.double() - h).abs().max() / h.abs().max()) <= 1e-5
    for a, b in zip(got, [x2.grad] + [p.grad for p in params]):
        assert float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-30)) <= 1e-4
