"""End-to-end engine tests on CPU: driver smoke runs (BASELINE.json config 1), parity of one
block visit against a literal reference-style loop, multi-process (gloo) == single-process."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import golden_data

from federated_pytorch_test_b200 import models
from federated_pytorch_test_b200.api import (consensus_multi, federated_cpc, federated_multi, federated_vae,
                                             federated_vae_cl, fedprox_multi, no_consensus_multi)

TINY = dict(train_size=1024, test_size=128, save_model=False, graphs=False, fast=False)


def _run(mod, **kw):
    lines = []
    eng = mod.run(mod.Config(**{**TINY, **kw}), log=lines.append)
    return eng, lines


def test_no_consensus_simplecnn_k2_cpu():
    """BASELINE.json config 1: no_consensus_multi SimpleCNN K=2 on CPU."""
    eng, lines = _run(no_consensus_multi, K=2, Nepoch=2, max_minibatches=4, check_results=True, use_cuda=False)
    assert lines[0] == "Epoch 0" and lines[-1] == "Finished Training"
    assert sum(l.startswith("Accuracy of the network") for l in lines) == 4
    assert eng.images_seen == 2 * 2 * 511  # shards of 1024/2 - 1 samples (Q1 off-by-one), 4 minibatches each


def test_federated_multi_blocks_and_writeback():
    eng, lines = _run(federated_multi, K=3, Nloop=1, Nadmm=2, max_minibatches=2, check_results=False, use_cuda=False)
    duals = [l for l in lines if l.startswith("dual (")]
    assert len(duals) == 5 * 2
    assert duals[0].startswith("dual (epoch=0,loop=0,block=[4,5],avg=0)=")
    # after FedAvg every replica holds identical parameters
    a, b = eng.replicas[0].arenas["net"].data, eng.replicas[2].arenas["net"].data
    torch.testing.assert_close(a, b)


def test_nan_in_one_replica_is_detected_at_the_next_aggregation():
    """Failure detection (SURVEY §5.3): a diverged replica poisons the reduced vector; every rank sees a non-finite
    residual at the next round and the engine stops with a message naming block and round (or warns)."""
    from federated_pytorch_test_b200.algo.engine import Engine

    def poison(e: Engine):
        if e.steps_done == 1:
            e.replicas[1].arenas["net"].data.fill_(float("nan"))

    for guard in ("raise", "warn"):
        lines = []
        cfg = federated_multi.Config(**{**TINY, **dict(K=2, Nloop=1, Nadmm=1, max_minibatches=1, check_results=False,
                                                       use_cuda=False, nan_guard=guard)})
        orig_init = Engine.__init__

        def patched(self, *a, **k):
            orig_init(self, *a, **k)
            self.step_hook = poison
        Engine.__init__ = patched
        try:
            if guard == "raise":
                with pytest.raises(FloatingPointError, match="non-finite dual residual after aggregating block"):
                    federated_multi.run(cfg, log=lines.append)
            else:
                federated_multi.run(cfg, log=lines.append)
                assert any(l.startswith("WARNING: non-finite dual residual") for l in lines)
        finally:
            Engine.__init__ = orig_init


def test_fedprox_and_consensus_do_not_write_back():
    eng, lines = _run(fedprox_multi, K=2, Nloop=1, Nadmm=2, max_minibatches=2, check_results=False, use_cuda=False)
    assert lines[0].startswith("block=[4,5](48120,1.000000) ADMM=0/0 primal=")
    assert not torch.allclose(eng.replicas[0].arenas["net"].data, eng.replicas[1].arenas["net"].data)
    eng, lines = _run(consensus_multi, K=2, Nloop=1, Nadmm=3, max_minibatches=2, check_results=False, use_cuda=False,
                      bb_update=True)
    assert any(l.startswith("admm 2 deltas=(") for l in lines)
    assert any(l.startswith("block=[8,9](850,") for l in lines)


def test_resnet_and_lbfgs_options():
    eng, lines = _run(federated_multi, K=2, Nloop=1, Nadmm=1, max_minibatches=1, check_results=False, use_cuda=False,
                      model="ResNet9", default_batch=8)
    assert len([l for l in lines if l.startswith("dual (")]) == 8
    eng, lines = _run(fedprox_multi, K=2, Nloop=1, Nadmm=1, max_minibatches=1, check_results=False, use_cuda=False,
                      optimizer="lbfgs", default_batch=16)
    assert len([l for l in lines if l.startswith("block=[")]) == 5


def test_vae_vaecl_cpc_drivers(tmp_path):
    eng, lines = _run(federated_vae, K=2, Nloop=1, Nadmm=1, max_minibatches=1, be_verbose=False, use_cuda=False)
    assert len([l for l in lines if l.startswith("dual (")]) == 12
    assert lines[0].startswith("dual (epoch=0,loop=0,block=[0,1],avg=0)=")
    eng, lines = _run(federated_vae_cl, K=2, Nloop=1, Nadmm=1, max_minibatches=1, be_verbose=True, use_cuda=False,
                      default_batch=8, Kc=3, Lc=4)
    assert any(l.startswith("cluster 2 costs ") for l in lines)
    assert [l for l in lines if l.startswith("dual (")][1].startswith("dual (epoch=0,loop=0,block=[32,41],avg=0)=")
    cfg = federated_cpc.Config(K=2, Lc=32, Rc=8, batch_size=2, Niter=1, load_model=False, init_model=True, save_model=True,
                               be_verbose=False, nbase=4, ckpt_dir=str(tmp_path), graphs=False, fast=False, use_cuda=False)
    lines = []
    federated_cpc.run(cfg, log=lines.append)
    assert len([l for l in lines if l.startswith("dual (N=")]) == 4
    assert sorted(os.listdir(tmp_path)) == ["contextgen0.model", "contextgen1.model", "encoder0.model", "encoder1.model",
                                            "predictor0.model", "predictor1.model"]


# ----------------------------------------------------------------------------------------------
K_VISIT, B_VISIT, STEPS_VISIT, ROUNDS_VISIT, RHO_VISIT, CI_VISIT, LAM1_VISIT, LAM2_VISIT = 2, 16, 3, 2, 0.1, 4, 1e-4, 1e-4


def _visit_data():
    g = torch.Generator().manual_seed(0)
    return {k: [(torch.randn(B_VISIT, 3, 32, 32, generator=g), torch.randint(0, 10, (B_VISIT,), generator=g))
                for _ in range(STEPS_VISIT)] for k in range(K_VISIT)}


def golden(ref):
    """The reference recipe of one ADMM block visit (torch.optim.Adam + autograd through torch.cat,
    get/put_trainable_values) on the reference's Net and utilities; see golden_data.py."""
    ref_models, ref_utils = ref.models, ref.utils
    K, steps, rounds, rho, ci, lam1, lam2 = K_VISIT, STEPS_VISIT, ROUNDS_VISIT, RHO_VISIT, CI_VISIT, LAM1_VISIT, LAM2_VISIT
    data = _visit_data()
    nets = {}
    for k in range(K):
        nets[k] = ref_models.Net()
        torch.manual_seed(0)
        nets[k].apply(ref_utils.init_weights)
        ref_utils.unfreeze_one_block(nets[k], ci)
    N = ref_utils.get_trainable_values(nets[0]).numel()
    z = torch.zeros(N)
    ys = {k: torch.zeros(N) for k in range(K)}
    opts = {k: torch.optim.Adam(filter(lambda p: p.requires_grad, nets[k].parameters()), lr=1e-3) for k in range(K)}
    ref_trace = []
    for r in range(rounds):
        for k in range(K):
            for xb, yb in data[k]:
                opts[k].zero_grad()
                vec = torch.cat([p.view(-1) for p in nets[k].parameters() if p.requires_grad])
                xd = vec - z
                loss = F.cross_entropy(nets[k](xb), yb) + torch.dot(ys[k], xd) + 0.5 * rho * torch.norm(xd, 2) ** 2
                loss = loss + lam1 * torch.norm(vec, 1) + lam2 * torch.norm(vec, 2) ** 2   # block 4 of Net is gated on
                loss.backward()
                opts[k].step()
        xs = {k: ref_utils.get_trainable_values(nets[k]) for k in range(K)}
        znew = sum(ys[k] + rho * xs[k] for k in range(K)) / (K * rho)
        dual = float(torch.norm(z - znew)) / N
        z = znew
        primal = 0.0
        for k in range(K):
            yd = rho * (xs[k] - z)
            primal += float(torch.norm(yd))
            ys[k].add_(yd)
        ref_trace.append((primal / N, dual))
    out = {"visit/trace": np.array(ref_trace)}
    for k in range(K):
        out.update(golden_data.digest(ref_utils.get_trainable_values(nets[k]), "visit/x%d" % k))
    return out


def test_block_visit_matches_reference_style_loop():
    """One ADMM block visit: BlockAdam + closed-form penalty on arena slices  ==  the reference recipe (``golden``
    above) on the same batches."""
    from federated_pytorch_test_b200.algo.engine import Engine, EngineConfig, Replica, Task, Visit
    from federated_pytorch_test_b200.algo.strategies import ADMM
    from federated_pytorch_test_b200.parallel import Topology, TorchCollective
    from federated_pytorch_test_b200.utils import init_weights

    K, rounds, rho, ci, lam1, lam2 = K_VISIT, ROUNDS_VISIT, RHO_VISIT, CI_VISIT, LAM1_VISIT, LAM2_VISIT
    data = _visit_data()
    g = golden_data.load("test_engine")
    ref_trace = [tuple(r) for r in g["visit/trace"]]

    class FixedTask(Task):
        def build_replica(self, ck, device, allocator):
            net = models.Net()
            rep = Replica(ck, {"net": net}, device)
            torch.manual_seed(0)
            net.apply(init_weights)
            return rep

        def visits(self, nloop):
            lo, hi = models.Net().train_order_block_ids()[ci]
            yield Visit("net", lo, hi, ci, (lo, hi), "adam", dict(lr=1e-3), lambda1=lam1, lambda2=lam2)

        def batches(self, rep, visit, epoch):
            return iter(data[rep.ck])

        def loss(self, rep, batch):
            return F.cross_entropy(rep.nets["net"](batch[0]), batch[1])

        def aggregate_log(self, visit, metrics, ctx, engine):
            trace.append((metrics["primal"], metrics["dual"]))

    trace = []
    topo = Topology.single_process(K, "cpu")
    coll = TorchCollective(topo)
    strat = ADMM(coll, topo, 5, rho0=rho)
    eng = Engine(FixedTask(), topo, strat, coll, EngineConfig(Nloop=1, Nadmm=rounds, Nepoch=1), log=lambda m: None)
    eng.run()
    assert len(trace) == len(ref_trace) == rounds
    for (p1, d1), (p2, d2) in zip(ref_trace, trace):
        assert p2 == pytest.approx(p1, rel=2e-3) and d2 == pytest.approx(d1, rel=2e-3)
    lo, hi = models.Net().train_order_block_ids()[ci]
    for k in range(K):
        mine = eng.replicas[k].arenas["net"].compact(lo, hi)
        golden_data.assert_matches(mine, g, "visit/x%d" % k, rtol=1e-3, atol=1e-5)


# ----------------------------------------------------------------------------------------------
def _dist_worker(rank, world, port, out):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    lines = []
    cfg = federated_multi.Config(K=2, Nloop=1, Nadmm=2, max_minibatches=2, check_results=False, use_cuda=False, **TINY)
    eng = federated_multi.run(cfg, log=lines.append)
    if rank == 0:
        torch.save({"lines": lines, "flat": eng.replicas[0].arenas["net"].data.clone()}, out)
    dist.destroy_process_group()


def test_two_process_gloo_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "r0.pt")
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_dist_worker, args=(2, port, out), nprocs=2, join=True)
    got = torch.load(out, weights_only=False)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        os.environ.pop(k, None)
    eng, lines = _run(federated_multi, K=2, Nloop=1, Nadmm=2, max_minibatches=2, check_results=False, use_cuda=False)
    single = [l for l in lines if l.startswith("dual (")]
    multi = [l for l in got["lines"] if l.startswith("dual (")]
    assert len(single) == len(multi) == 10
    for a, b in zip(single, multi):
        assert a.split("=")[:-1] == b.split("=")[:-1]
        assert float(a.rsplit("=", 1)[1]) == pytest.approx(float(b.rsplit("=", 1)[1]), rel=1e-4)
    torch.testing.assert_close(got["flat"], eng.replicas[0].arenas["net"].data, rtol=1e-4, atol=1e-6)


def _coresident_worker(rank, world, port, out, K, algo):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    mod = federated_multi if algo == "fedavg" else consensus_multi
    extra = {} if algo == "fedavg" else dict(bb_update=True)
    lines = []
    cfg = mod.Config(K=K, Nloop=1, Nadmm=2, max_minibatches=2, check_results=False, use_cuda=False, **TINY, **extra)
    eng = mod.run(cfg, log=lines.append)
    if rank == 0:
        torch.save({"lines": lines, "local": [r.ck for r in eng.replicas]}, out)
    dist.destroy_process_group()


@pytest.mark.parametrize("algo", ["fedavg", "admm"])
def test_co_resident_replicas_over_two_ranks_match_single_process(tmp_path, algo):
    """K = 4 workers on 2 processes (two co-resident replicas per rank, gloo): same residual trace as the
    single-process K = 4 run — the K > #GPUs placement of SURVEY §2.8, including the Barzilai-Borwein rho replay."""
    import torch.multiprocessing as mp
    out = str(tmp_path / "r0.pt")
    port = 31500 + (os.getpid() % 2000) + (11 if algo == "admm" else 0)
    mp.spawn(_coresident_worker, args=(2, port, out, 4, algo), nprocs=2, join=True)
    got = torch.load(out, weights_only=False)
    assert got["local"] == [0, 2]
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        os.environ.pop(k, None)
    mod = federated_multi if algo == "fedavg" else consensus_multi
    extra = {} if algo == "fedavg" else dict(bb_update=True)
    _, lines = _run(mod, K=4, Nloop=1, Nadmm=2, max_minibatches=2, check_results=False, use_cuda=False, **extra)
    key = "dual (" if algo == "fedavg" else "block=["
    a = [l for l in got["lines"] if l.startswith(key)]
    b = [l for l in lines if l.startswith(key)]
    assert len(a) == len(b) == 10
    for x, y in zip(a, b):
        assert float(x.rsplit("=", 1)[1]) == pytest.approx(float(y.rsplit("=", 1)[1]), rel=1e-3, abs=1e-9), (x, y)


# ------------------------------------------------------------------------------------------ true resume (SURVEY §5.4)
class _Killed(Exception):
    pass


@pytest.mark.parametrize("mod,extra", [(fedprox_multi, {}), (consensus_multi, {"bb_update": True}), (federated_multi, {})])
def test_kill_and_resume_reproduces_the_trace(tmp_path, mod, extra):
    """Run A: uninterrupted.  Run B: killed mid-schedule (inside a block visit, between two rounds), then a NEW process
    state (fresh engine) resumes from the record the engine wrote after the last completed round.  The residual traces
    of B-before + B-after must equal A line by line: schedule position, z / y / rho / BB vectors, Adam moments + step
    count, loader RNG and global RNG all re-enter exactly."""
    from federated_pytorch_test_b200.algo.engine import Engine

    kw = dict(K=2, Nloop=1, Nadmm=3, max_minibatches=2, check_results=False, use_cuda=False, **extra)
    key = "dual (" if mod is federated_multi else "block=["
    _, full = _run(mod, **kw)
    full = [l for l in full if l.startswith(key)]
    assert len(full) == 15

    rec = str(tmp_path / "resume.pt")
    kill_at = 2 * 2 * (3 + 2) - 1          # a step inside round 2 of the second block visit (7 rounds completed before it... )
    orig_init = Engine.__init__

    def patched(self, *a, **k):
        orig_init(self, *a, **k)

        def hook(e):
            if e.steps_done == kill_at:
                raise _Killed()
        self.step_hook = hook
    Engine.__init__ = patched
    first = []
    try:
        with pytest.raises(_Killed):
            mod.run(mod.Config(**{**TINY, **kw, "resume_out": rec}), log=first.append)
    finally:
        Engine.__init__ = orig_init
    first = [l for l in first if l.startswith(key)]
    assert 0 < len(first) < 15 and os.path.exists(rec)
    _, second = _run(mod, **kw, resume=rec)
    second = [l for l in second if l.startswith(key)]
    assert first + second == full
