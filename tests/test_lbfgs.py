"""LBFGSNew against the reference implementation (SURVEY §2.5, §4)."""
import warnings

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

import golden_data

from federated_pytorch_test_b200.optim import LBFGSNew
from federated_pytorch_test_b200.utils import FlatArena

warnings.filterwarnings("ignore")


def _rosenbrock(cls):
    x = nn.Parameter(torch.tensor([-1.2, 1.0]))
    opt = cls([x], history_size=7, max_iter=100, line_search_fn=True, batch_mode=False)
    calls = [0]

    def closure():
        calls[0] += 1
        if torch.is_grad_enabled():
            opt.zero_grad()
        f = (1 - x[0]) ** 2 + 100 * (x[1] - x[0] ** 2) ** 2
        if f.requires_grad:
            f.backward()
        return f

    opt.step(closure)
    st = opt.state[opt._params[0]]
    return x.detach().clone(), calls[0], st["n_iter"], st["func_evals"]


def test_rosenbrock_golden():
    x, calls, iters, evals = _rosenbrock(LBFGSNew)
    torch.testing.assert_close(x, torch.tensor([1.0, 1.0]), atol=1e-5, rtol=0)
    assert (calls, iters) == (655, 31)  # BASELINE.md §2


def test_rosenbrock_identical_to_reference():
    g = golden_data.load("test_lbfgs")
    x, *counts = _rosenbrock(LBFGSNew)
    assert torch.equal(x, torch.from_numpy(g["rosenbrock/x"])) and counts == g["rosenbrock/counts"].tolist()


def _stochastic(cls, arena=False, steps=5):
    """Five stochastic L-BFGS steps on one CPU thread: the iterates are compared bit for bit with stored values, and
    the convolution's weight gradient is a reduction whose rounding depends on how many threads share it."""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        return _stochastic_run(cls, arena, steps)
    finally:
        torch.set_num_threads(threads)


def _stochastic_run(cls, arena, steps):
    torch.manual_seed(0)
    net = nn.Sequential(nn.Conv2d(3, 8, 3), nn.ELU(), nn.Flatten(), nn.Linear(8 * 30 * 30, 10))
    if arena:
        FlatArena(net).attach_grads()
    opt = cls(net.parameters(), history_size=10, max_iter=4, line_search_fn=True, batch_mode=True)
    g = torch.Generator().manual_seed(1)
    log = []
    for _ in range(steps):
        xb, yb = torch.randn(32, 3, 32, 32, generator=g), torch.randint(0, 10, (32,), generator=g)
        cnt = [0, 0]

        def closure():
            if torch.is_grad_enabled():
                opt.zero_grad()
            loss = F.cross_entropy(net(xb), yb)
            cnt[0] += 1
            if loss.requires_grad:
                loss.backward()
                cnt[1] += 1
            return loss

        loss = opt.step(closure)
        log.append((float(loss), cnt[0], cnt[1]))
    vec = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
    return log, vec, opt


def golden(ref):
    """The reference's LBFGSNew on the two problems above; see golden_data.py."""
    x, *counts = _rosenbrock(ref.lbfgs.LBFGSNew)
    log, vec, opt = _stochastic(ref.lbfgs.LBFGSNew)
    return {"rosenbrock/x": x.numpy(), "rosenbrock/counts": np.array(counts),
            "stochastic/counts": np.array([x[1:] for x in log]), "stochastic/sha256": np.array(golden_data.sha256(vec)),
            "stochastic/state_keys": np.array(sorted(opt.state_dict()["state"][0].keys()))}


def test_stochastic_identical_to_reference():
    g = golden_data.load("test_lbfgs")
    log, vec, opt = _stochastic(LBFGSNew)
    assert [list(x[1:]) for x in log] == g["stochastic/counts"].tolist()       # forward/backward counts per step
    assert golden_data.sha256(vec) == str(g["stochastic/sha256"])             # bit-identical iterates
    assert sorted(opt.state_dict()["state"][0].keys()) == list(g["stochastic/state_keys"])


def test_stochastic_on_arena_close_to_reference():
    g = golden_data.load("test_lbfgs")
    a, c = _stochastic(LBFGSNew), _stochastic(LBFGSNew, arena=True)
    assert golden_data.sha256(a[1]) == str(g["stochastic/sha256"])            # a is the reference's result, bit for bit
    assert [list(x[1:]) for x in c[0]] == g["stochastic/counts"].tolist()
    torch.testing.assert_close(a[1], c[1], rtol=1e-4, atol=1e-5)
    assert c[2]._v().fused


def test_state_dict_roundtrip():
    _, _, opt = _stochastic(LBFGSNew, steps=3)
    sd = opt.state_dict()
    assert "_hist" not in sd["state"][0]
    assert len(sd["state"][0]["old_dirs"]) > 0
    assert "_hist" in opt.state[opt._params[0]]  # live state untouched
