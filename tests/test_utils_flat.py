"""simple_utils API + flat arena (SURVEY §2.3, §4 unit level)."""
import numpy as np
import pytest
import torch
import torch.nn as nn

import golden_data

from federated_pytorch_test_b200 import models
from federated_pytorch_test_b200.utils import (FlatArena, freeze_all_layers, get_trainable_values, init_weights,
                                               number_of_blocks, number_of_layers, put_trainable_values,
                                               unfreeze_all_layers, unfreeze_one_block, unfreeze_one_layer)

ALL = [models.Net, models.Net1, models.Net2, models.ResNet9, models.AutoEncoderCNN,
       lambda: models.AutoEncoderCNNCL(4, 8), lambda: models.EncoderCNN(32), lambda: models.ContextgenCNN(32),
       lambda: models.PredictorCNN(32, 8)]


@pytest.mark.parametrize("factory", ALL)
@pytest.mark.parametrize("use_arena", [False, True])
def test_block_masks_and_roundtrip(factory, use_arena):
    net = factory()
    if use_arena:
        FlatArena(net)
    n = number_of_layers(net)
    assert n == len(list(net.parameters()))
    for b, (lo, hi) in enumerate(net.train_order_block_ids()):
        unfreeze_one_block(net, b)
        flags = [p.requires_grad for p in net.parameters()]
        assert flags == [lo <= i <= hi for i in range(n)]
        v = get_trainable_values(net)
        assert v.numel() == sum(p.numel() for i, p in enumerate(net.parameters()) if lo <= i <= hi)
        w = torch.randn_like(v)
        put_trainable_values(net, w)
        torch.testing.assert_close(get_trainable_values(net), w)
    assert number_of_blocks(net) == len(net.train_order_block_ids())
    unfreeze_all_layers(net)
    assert all(p.requires_grad for p in net.parameters())
    freeze_all_layers(net)
    assert not any(p.requires_grad for p in net.parameters())
    unfreeze_one_layer(net, 0)
    assert [p.requires_grad for p in net.parameters()][:3] == [True, True, False][: min(3, n)]


def _packed(m, unfreeze, get_values, arena=False):
    """get_trainable_values of every block of Net (seeded weights), block after block."""
    net = golden_data.fill_(m.Net(), seed=13)
    if arena:
        FlatArena(net)
    out = []
    for b in range(5):
        unfreeze(net, b)
        out.append(get_values(net))
    return out


def _initialised(m, init, arena=False):
    net = m.ResNet9()
    if arena:
        FlatArena(net, channels_last_weights=True)   # values must not depend on the memory format
    torch.manual_seed(0)
    net.apply(init)
    return net


def golden(ref):
    """What the reference computes in the comparisons below (see golden_data.py)."""
    out = {}
    for b, v in enumerate(_packed(ref.models, ref.utils.unfreeze_one_block, ref.utils.get_trainable_values)):
        out.update(golden_data.digest(v, "pack/%d" % b))
    sd = _initialised(ref.models, ref.utils.init_weights).state_dict()
    out["init/keys"] = np.array(list(sd))
    for k, v in sd.items():
        out.update(golden_data.digest(v, "init/" + k, k=64))
    return out


def test_pack_matches_reference():
    g = golden_data.load("test_utils_flat")
    for b, v in enumerate(_packed(models, unfreeze_one_block, get_trainable_values, arena=True)):
        golden_data.assert_matches(v, g, "pack/%d" % b)


def test_init_weights_matches_reference():
    g = golden_data.load("test_utils_flat")
    sd = _initialised(models, init_weights, arena=True).state_dict()
    assert list(sd) == list(g["init/keys"])
    for k, a in sd.items():
        golden_data.assert_matches(a.contiguous(), g, "init/" + k)
    # ConvTranspose2d untouched (Q15): default init differs from xavier, bias not 0.01
    vae = models.AutoEncoderCNN()
    vae.apply(init_weights)
    assert not torch.allclose(vae.tconv1.bias, torch.full_like(vae.tconv1.bias, 0.01))
    assert torch.allclose(vae.conv1.bias, torch.full_like(vae.conv1.bias, 0.01))


def test_arena_views_and_alignment():
    net = models.Net()
    ref = [p.detach().clone() for p in net.parameters()]
    arena = FlatArena(net, align=32)
    assert arena.check_views()
    for p, r, off in zip(net.parameters(), ref, arena.offsets):
        torch.testing.assert_close(p.detach(), r)
        assert off % 32 == 0
    # a block is a contiguous slice and updates through the slice are visible in the parameters
    lo, hi = net.train_order_block_ids()[0]
    sl = arena.block(lo, hi)
    sl.zero_()
    assert float(net.fc1.weight.abs().sum()) == 0.0 and float(net.fc1.bias.abs().sum()) == 0.0
    assert arena.count(lo, hi) == 48120
    # gradients accumulate into the gradient arena without breaking the views
    unfreeze_one_block(net, 0)
    out = net(torch.randn(2, 3, 32, 32)).sum()
    out.backward()
    assert net.fc1.weight.grad.data_ptr() == arena.grad_view(4).data_ptr()
    assert float(arena.block_grad(lo, hi).abs().sum()) > 0
    assert net.conv1.weight.grad is None


def test_arena_channels_last_and_state_dict_roundtrip(tmp_path):
    from federated_pytorch_test_b200.utils import ckpt
    net = models.ResNet9()
    before = {k: v.clone() for k, v in net.state_dict().items()}
    arena = FlatArena(net, channels_last_weights=True)
    assert net.conv1.weight.is_contiguous(memory_format=torch.channels_last)
    for k, v in net.state_dict().items():
        torch.testing.assert_close(v.contiguous(), before[k])
    dense = ckpt.dense_state_dict(net)
    assert all(t.is_contiguous() for t in dense.values())
    other = models.ResNet9()
    FlatArena(other)
    ckpt.load_into(other, dense)
    x = torch.randn(2, 3, 32, 32)
    torch.testing.assert_close(other(x), net(x), rtol=1e-4, atol=1e-4)
    assert arena.check_views() and other._flat_arena.check_views()
