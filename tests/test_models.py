"""Model zoo: shapes, parameter/block inventory (SURVEY §2.2) and forward parity with the reference."""
import numpy as np
import pytest
import torch

import golden_data

from federated_pytorch_test_b200 import models
from federated_pytorch_test_b200.ops import functional as FX

SPEC = [  # (factory, #tensors, #params)
    (models.Net, 10, 62006), (models.Net1, 12, 890410), (models.Net2, 18, 2513418),
    (models.ResNet18, 62, 11173962), (models.ResNet9, 38, 4903242),
    (models.AutoEncoderCNN, 24, 205679), (lambda: models.AutoEncoderCNNCL(10, 32), 42, 350744),
    (lambda: models.EncoderCNN(256), 16, 701928), (lambda: models.ContextgenCNN(256), 4, 98304),
    (lambda: models.PredictorCNN(256, 32), 2, 16384),
]


@pytest.mark.parametrize("factory,ntensors,nparams", SPEC)
def test_inventory(factory, ntensors, nparams):
    net = factory()
    ps = list(net.parameters())
    assert len(ps) == ntensors
    assert sum(p.numel() for p in ps) == nparams
    covered = []
    for lo, hi in net.train_order_block_ids():
        covered += list(range(lo, hi + 1))
    assert sorted(covered) == list(range(ntensors)), "blocks must cover every parameter index exactly once"


def test_resnet18_block_sizes():
    net = models.ResNet18()
    sizes = [net.block_numel(i) for i in range(10)]
    assert sizes == [1856, 73984, 73984, 230144, 295424, 919040, 1180672, 3673088, 4720640, 5130]
    assert [models.Net().block_numel(i) for i in range(5)] == [48120, 456, 2416, 10164, 850]


def test_protocol_methods():
    net = models.Net()
    assert net.linear_layer_ids() == [4, 6, 8]
    assert net.train_order_block_ids() == [[4, 5], [0, 1], [2, 3], [6, 7], [8, 9]]
    assert net.linear_layer_parameters().numel() == 48120 + 10164 + 850
    assert models.ResNet18().linear_layer_ids() == []


PAIRS = [("Net", lambda m: m.Net(), (4, 3, 32, 32)), ("Net1", lambda m: m.Net1(), (4, 3, 32, 32)),
         ("Net2", lambda m: m.Net2(), (4, 3, 32, 32)), ("ResNet18", lambda m: m.ResNet18(), (4, 3, 32, 32)),
         ("ResNet9", lambda m: m.ResNet9(), (4, 3, 32, 32)),
         ("ContextgenCNN", lambda m: m.ContextgenCNN(32), (2, 32, 3, 3))]


def _layout(name, net):
    sd = net.state_dict()
    return {name + "/keys": np.array(list(sd)), name + "/shapes": np.array([",".join(map(str, t.shape)) for t in sd.values()])}


def _forward(m, make, shape):
    """``make(m)`` with the seeded weights of ``golden_data.fill_`` and its output on a seeded input."""
    FX.set_fast_path(False)
    net = golden_data.fill_(make(m))
    return net, net(golden_data.randn(*shape, seed=1))


def _encoder_predictor(m):
    enc = golden_data.fill_(m.EncoderCNN(64), seed=2)
    pred = golden_data.fill_(m.PredictorCNN(64, 8), seed=3)
    y = enc(golden_data.randn(6, 8, 32, 32, seed=4))
    return enc, pred, [y] + list(pred(golden_data.randn(2, 64, 3, 3, seed=5), golden_data.randn(2, 64, 3, 3, seed=6)))


def _uniform(*shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


def _vae(m):
    net = golden_data.fill_(m.AutoEncoderCNN(), seed=7)
    return net, list(net.encode(_uniform(3, 3, 32, 32, seed=8))) + [net.decode(golden_data.randn(3, 10, seed=9))]


_EK = torch.zeros(5, 4)
_EK[:, 2] = 1


def _vae_cl_heads(net):
    """encodeclus, then the deterministic heads of cluster 2 (encode, decode)."""
    x = _uniform(5, 3, 32, 32, seed=11)
    return [net.encodeclus(x)], list(net.encode(x, _EK)), list(net.decode(_EK, golden_data.randn(5, 8, seed=12)))


def golden(ref):
    """What the reference computes in the comparisons below (see golden_data.py)."""
    out = {}
    for name, make, shape in PAIRS:
        net, y = _forward(ref.models, make, shape)
        out.update(_layout(name, net), **golden_data.digest(y, name + "/out"))
    enc, pred, ys = _encoder_predictor(ref.models)
    out.update(_layout("EncoderCNN", enc), **_layout("PredictorCNN", pred))
    for i, y in enumerate(ys):
        out.update(golden_data.digest(y, "encoder_predictor/%d" % i))
    net, ys = _vae(ref.models)
    out.update(_layout("AutoEncoderCNN", net))
    for i, y in enumerate(ys):
        out.update(golden_data.digest(y, "vae/%d" % i))
    net = golden_data.fill_(ref.models.AutoEncoderCNNCL(K=4, L=8), seed=10)
    out.update(_layout("AutoEncoderCNNCL", net))
    for part, ys in zip(("encodeclus", "encode", "decode"), _vae_cl_heads(net)):
        for i, y in enumerate(ys):
            out.update(golden_data.digest(y, "vae_cl/%s/%d" % (part, i)))
    return out


def _check_layout(name, net):
    g = golden_data.load("test_models")
    mine = _layout(name, net)
    assert list(mine[name + "/keys"]) == list(g[name + "/keys"]) and list(mine[name + "/shapes"]) == list(g[name + "/shapes"])


@pytest.mark.parametrize("name,make,shape", PAIRS)
def test_forward_matches_reference(name, make, shape):
    """Same state_dict layout as the reference, and the reference's outputs when given the same weights."""
    net, y = _forward(models, make, shape)
    _check_layout(name, net)
    golden_data.assert_matches(y, golden_data.load("test_models"), name + "/out", rtol=1e-5, atol=1e-5)


def test_encoder_predictor_match_reference():
    enc, pred, ys = _encoder_predictor(models)
    _check_layout("EncoderCNN", enc)
    _check_layout("PredictorCNN", pred)
    g = golden_data.load("test_models")
    assert len([k for k in g if k.startswith("encoder_predictor/") and k.endswith("/shape")]) == len(ys)
    golden_data.assert_matches(ys[0], g, "encoder_predictor/0", rtol=1e-5, atol=1e-5)
    for i, y in enumerate(ys[1:], 1):
        golden_data.assert_matches(y, g, "encoder_predictor/%d" % i)


def test_vae_deterministic_parts_match_reference():
    net, ys = _vae(models)
    _check_layout("AutoEncoderCNN", net)
    g = golden_data.load("test_models")
    assert len([k for k in g if k.startswith("vae/") and k.endswith("/shape")]) == len(ys)
    for i, y in enumerate(ys):
        golden_data.assert_matches(y, g, "vae/%d" % i, rtol=1e-5, atol=1e-6)


def test_vae_cl_batched_equals_loop():
    a = golden_data.fill_(models.AutoEncoderCNNCL(K=4, L=8, batched_clusters=True), seed=10)
    b = golden_data.fill_(models.AutoEncoderCNNCL(K=4, L=8, batched_clusters=False), seed=10)
    _check_layout("AutoEncoderCNNCL", a)
    a.force_disable_repr()
    b.force_disable_repr()
    # encodeclus and the deterministic heads against the reference, cluster by cluster
    g = golden_data.load("test_models")
    for part, ys in zip(("encodeclus", "encode", "decode"), _vae_cl_heads(a)):
        assert len([k for k in g if k.startswith("vae_cl/%s/" % part) and k.endswith("/shape")]) == len(ys)
        for i, y in enumerate(ys):
            golden_data.assert_matches(y, g, "vae_cl/%s/%d" % (part, i), rtol=1e-5, atol=1e-6)
    x = _uniform(5, 3, 32, 32, seed=11)
    oa, ob = a(x), b(x)
    torch.testing.assert_close(oa[0], ob[0])
    for da, db in zip(oa[1:], ob[1:]):
        for k in range(4):
            torch.testing.assert_close(da[k], db[k], rtol=1e-5, atol=1e-6)


def test_disable_repr_quirk_preserved():
    net = models.AutoEncoderCNNCL(2, 4)
    net.disable_repr()
    assert net.repr_flag is True  # SURVEY Q11
    net.force_disable_repr()
    assert net.repr_flag is False
