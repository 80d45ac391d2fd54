"""CPU tests of the host-side logic added late in round 2: the split aggregate_begin / aggregate_end protocol (deferred
rounds), the TF32-rounding fp64 oracle, the benchmark's window placement and the CPU fall-backs of the new fused ops."""
import importlib.util
import math
import os
import types

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from federated_pytorch_test_b200.algo.strategies import ADMM, FedAvg, FedProx
from federated_pytorch_test_b200.ops import functional as FX
from federated_pytorch_test_b200.parallel import Topology, TorchCollective
from federated_pytorch_test_b200.utils.tf32_oracle import tf32_conv_oracle, to_tf32

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _AsyncCollective(TorchCollective):
    """TorchCollective with the asynchronous entry points of FusedCollective: launch now, read the record later."""

    supports_async = True

    def __init__(self, topo):
        super().__init__(topo)
        self._rec = None
        self.reads = 0

    def launch_fedavg_(self, xs, z, write_back=True):
        self._rec = [self.fedavg_(xs, z, write_back=write_back), 0.0]

    def launch_fedprox_(self, xs, z, rho):
        self._rec = list(self.fedprox_(xs, z, rho))

    def launch_admm_(self, xs, ys, z, rho, rho_dev=None):
        self._rec = list(self.admm_(xs, ys, z, rho, rho_dev))

    def read_record(self):
        self.reads += 1
        return self._rec + [0.0] * 5


def _xs(K=4, N=257, seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(N, generator=g) for _ in range(K)]


@pytest.mark.parametrize("make", [lambda c, t: FedAvg(c, t), lambda c, t: FedProx(c, t, num_blocks=2, rho0=1.5),
                                  lambda c, t: ADMM(c, t, num_blocks=2, rho0=0.1)])
def test_split_aggregation_equals_synchronous(make):
    topo = Topology.single_process(4, "cpu")
    out = []
    for coll_cls in (TorchCollective, _AsyncCollective):
        xs = _xs()
        coll = coll_cls(topo)
        s = make(coll, topo)
        s.begin_block(0, 257, xs)
        rounds = []
        for nadmm in range(3):
            tok = s.aggregate_begin(nadmm)
            assert tok[0] == ("pending" if coll_cls is _AsyncCollective else "done")
            for x in xs:                       # the next minibatch runs before the record is read
                x.add_(0.01)
            rounds.append(s.aggregate_end(tok))
        if coll_cls is _AsyncCollective:
            assert coll.reads == 3
        out.append((rounds, [x.clone() for x in xs]))
    (ra, xa), (rb, xb) = out
    for ma, mb in zip(ra, rb):
        assert set(ma) == set(mb)
        for k in ma:
            assert ma[k] == pytest.approx(mb[k], rel=1e-6, abs=1e-12)
    for u, v in zip(xa, xb):
        torch.testing.assert_close(u, v)


def test_tf32_rounding_and_oracle():
    t = torch.tensor([1.0 + 2 ** -11 + 2 ** -20, 1.0 + 2 ** -10, -1.0 - 2 ** -11, 3.14159265], dtype=torch.float64)
    assert to_tf32(t, "trunc").tolist() == [1.0, 1.0 + 2 ** -10, -1.0, 3.140625]
    assert to_tf32(t, "rna").tolist() == [1.0 + 2 ** -10, 1.0 + 2 ** -10, -1.0 - 2 ** -10, 3.140625]
    torch.manual_seed(0)
    a = nn.Sequential(nn.Conv2d(3, 4, 3, padding=1), nn.ELU(), nn.Conv2d(4, 2, 3, padding=1)).double()
    b = nn.Sequential(nn.Conv2d(3, 4, 3, padding=1), nn.ELU(), nn.Conv2d(4, 2, 3, padding=1)).double()
    b.load_state_dict(a.state_dict())
    tf32_conv_oracle(b, "rna")
    x = torch.randn(2, 3, 8, 8, dtype=torch.float64)
    xa, xb = x.clone().requires_grad_(), x.clone().requires_grad_()
    a(xa).square().sum().backward()
    b(xb).square().sum().backward()
    rel = lambda u, v: float((u - v).abs().max() / u.abs().max())
    errs = [rel(xa.grad, xb.grad)] + [rel(p.grad, q.grad) for p, q in zip(a.parameters(), b.parameters())]
    assert all(1e-6 < e < 1e-2 for e in errs[:-1]), errs        # TF32-sized differences, not zero and not garbage
    assert errs[-1] < 1e-2                                        # last bias: sum of dy, rounded only through dy's dependence


def _bench():
    spec = importlib.util.spec_from_file_location("_bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def test_bench_windows_straddle_the_second_and_a_later_boundary():
    b = _bench()
    spr = b.STEPS_PER_ROUND
    assert b.TIMED_BOUNDARY == 2 * spr
    for K, W in ((20, 5), (40, 5), (10, 3), (2, 3), (100, 5), (200, 10)):
        first = b.straddle_window(K, W, b.PRIME_STEPS, b.TIMED_BOUNDARY)
        last = first + K
        assert first >= b.PRIME_STEPS + W                         # at least W warm-up steps after the priming steps
        assert first <= b.TIMED_BOUNDARY - 1 and last >= b.TIMED_BOUNDARY + 1     # steps 97 and 98 inside: the aggregation between them is timed
        if K < b.TIMED_BOUNDARY:
            assert first >= spr                                   # the first aggregation of the run is warm-up
        b_host = -(-last // spr) * spr
        fe = b.straddle_window(K, W, b_host, b_host + spr)
        assert fe >= b_host + min(W, spr) or K >= 2 * spr
        assert fe <= b_host + spr - 1 and fe + K >= b_host + spr + 1


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs: the last step's loss and every state_dict entry of the trained model, float32 / float64 .npy."""
    torch.manual_seed(0)
    net = nn.Sequential(nn.Conv2d(3, 4, 3), nn.BatchNorm2d(4))
    net(torch.randn(2, 3, 8, 8))
    eng = types.SimpleNamespace(last_loss1=torch.tensor(0.25), replicas=[types.SimpleNamespace(nets={"net": net})])
    _bench().dump_outputs(str(tmp_path), eng)
    sd = net.state_dict()
    assert sorted(os.listdir(tmp_path)) == sorted(["loss.npy"] + ["net.%s.npy" % k for k in sd])
    assert np.load(tmp_path / "loss.npy").tolist() == [0.25]
    for k, v in sd.items():
        a = np.load(tmp_path / ("net.%s.npy" % k))
        assert a.dtype in (np.float32, np.float64) and a.shape == tuple(v.shape)
        assert np.array_equal(a, v.double().numpy())


def test_dilated_stem_and_tiny_map_conv_cpu_fallback():
    torch.manual_seed(1)
    convs = [nn.Conv2d(8, 8, 4, stride=2, dilation=d, padding=(3 * d) // 2) for d in (1, 2, 4, 8, 16)]
    x = torch.randn(3, 8, 32, 32)
    y = FX.dilated_stem(x, convs)
    ref = torch.cat([F.elu(c(x)) for c in convs], 1)
    assert y.shape == (3, 40, 16, 16)
    torch.testing.assert_close(y, ref)
    # im2col rows used by the GPU path of the tiny-map convolutions == F.unfold
    xc, k, p = torch.randn(3, 5, 4, 4), 2, 1
    xp = F.pad(xc, (p, p, p, p))
    rows = xp.unfold(2, k, 1).unfold(3, k, 1).permute(0, 2, 3, 1, 4, 5).reshape(3 * 25, 5 * 4)
    assert torch.equal(rows, F.unfold(xc, (k, k), padding=p).transpose(1, 2).reshape(3 * 25, 20))


def test_engine_deferred_rounds_same_trace_as_synchronous(monkeypatch):
    """The engine's deferred-round protocol end to end (CPU, a collective with the asynchronous entry points of FusedCollective):
    the record of a round is read after the next minibatch has been queued, the last round of a visit is finished at the visit's
    end — same log lines in the same order, same parameters as the synchronous engine."""
    from federated_pytorch_test_b200.api import common, federated_multi, fedprox_multi

    tiny = dict(train_size=1024, test_size=128, save_model=False, graphs=False, fast=False, use_cuda=False, check_results=False)
    for mod in (federated_multi, fedprox_multi):
        traces = []
        for cls in (TorchCollective, _AsyncCollective):
            made = []

            def make(topo, kind, _cls=cls):
                made.append(_cls(topo))
                return made[-1]

            monkeypatch.setattr(common, "make_collective", make)
            lines = []
            eng = mod.run(mod.Config(K=3, Nloop=1, Nadmm=3, max_minibatches=2, **tiny), log=lines.append)
            assert eng._pending_round is None
            if cls is _AsyncCollective:
                assert made[0].reads == eng.aggregations_done == 5 * 3
            traces.append(([l for l in lines if l.startswith(("dual (", "block=["))], eng.replicas[1].arenas["net"].data.clone()))
        (la, xa), (lb, xb) = traces
        assert len(la) == 15 and la == lb
        torch.testing.assert_close(xa, xb)
