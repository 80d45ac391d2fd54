"""Config/CLI (SURVEY §5.6), legacy checkpoints (§5.4) and log formats (§5.5)."""
import os

import torch

import golden_data

from federated_pytorch_test_b200 import models
from federated_pytorch_test_b200.config import (CPCConfig, ConsensusConfig, FedProxConfig, FederatedConfig,
                                                NoConsensusConfig, VAECLConfig, parse_config)
from federated_pytorch_test_b200.utils import FlatArena, ckpt, legacy_log


def test_defaults_match_reference_constants():
    f = FederatedConfig()
    assert (f.K, f.default_batch, f.Nloop, f.Nepoch, f.Nadmm, f.lambda1, f.lambda2) == (10, 128, 12, 1, 3, 1e-4, 1e-4)
    assert (f.load_model, f.init_model, f.save_model, f.check_results, f.biased_input, f.use_resnet) == (False, True, True, True, True, False)
    assert FedProxConfig().admm_rho0 == 1.0 and FedProxConfig().Nadmm == 5
    c = ConsensusConfig()
    assert (c.admm_rho0, c.Nadmm, c.bb_update, c.bb_period_T, c.bb_alphacorrmin, c.bb_epsilon, c.bb_rhomax) == (0.1, 5, False, 2, 0.2, 1e-3, 0.1)
    assert NoConsensusConfig().Nepoch == 20
    v = VAECLConfig()
    assert (v.K, v.Kc, v.Lc, v.lambda2) == (1, 10, 32, 1e-3)
    p = CPCConfig()
    assert (p.K, p.Lc, p.Rc, p.batch_size, p.Niter, p.load_model, p.init_model) == (4, 256, 32, 128, 10, True, False)


def test_cli_overrides():
    c = parse_config(ConsensusConfig, ["--K", "8", "--use_resnet", "--bb_update", "--no-check_results", "--admm_rho0", "0.05"])
    assert c.K == 8 and c.use_resnet and c.bb_update and not c.check_results and c.admm_rho0 == 0.05
    c = parse_config(FederatedConfig, ["--use_resnet=false", "--Nloop", "2"])
    assert c.use_resnet is False and c.Nloop == 2


def test_legacy_checkpoint_interop(tmp_path):
    g = golden_data.load("test_models")          # the reference's Net: state_dict layout, output with seeded weights
    layout = dict(zip(g["Net/keys"], g["Net/shapes"]))
    net = golden_data.fill_(models.Net())
    FlatArena(net)
    opt = torch.optim.Adam(net.parameters())
    path = ckpt.save_worker(str(tmp_path), 3, net, 0, opt, 1.25)
    assert os.path.basename(path) == "s3.model"
    blob = torch.load(path, weights_only=False)
    assert sorted(blob) == ["epoch", "model_state_dict", "optimizer_state_dict", "running_loss"]
    # the reference can read our file: its strict load_state_dict needs these keys and shapes, and the values it
    # loads are the seeded weights, on which it computes the stored output
    sd = blob["model_state_dict"]
    assert {k: ",".join(map(str, v.shape)) for k, v in sd.items()} == layout
    seeded = golden_data.fill_(models.Net()).state_dict()
    for k, v in sd.items():
        assert torch.equal(v, seeded[k]), k
    golden_data.assert_matches(net(golden_data.randn(4, 3, 32, 32, seed=1)), g, "Net/out")
    gen = torch.Generator().manual_seed(5)
    ref_sd = {k: torch.randn(*(int(d) for d in shape.split(",") if d), generator=gen) for k, shape in layout.items()}
    torch.save({"model_state_dict": ref_sd, "epoch": 0, "optimizer_state_dict": {}, "running_loss": 0.0},
               ckpt.worker_path(str(tmp_path), 4))
    ckpt.load_worker(str(tmp_path), 4, net, "cpu")          # and we can read the reference's
    assert net._flat_arena.check_views() and net.training
    for k, v in net.state_dict().items():
        assert torch.equal(v, ref_sd[k]), k


def test_log_formats_golden():
    assert legacy_log.accuracy_line(0, 10000, 900) == "Accuracy of the network 0 on the 10000 test images:%9.000000"
    assert legacy_log.dual_line(0, 0, (4, 5), 0, 2.820972e-04) == "dual (epoch=0,loop=0,block=[4,5],avg=0)=2.820972e-04"
    assert legacy_log.admm_line((4, 5), 48120, 0.095266, 4, 0, 2.639425e-07, 5.101571e-06) == \
        "block=[4,5](48120,0.095266) ADMM=4/0 primal=2.639425e-07 dual=5.101571e-06"
    assert legacy_log.minibatch_line(1, (0, 2), 3, 1856, 7, 0, 0.5) == "model=1 block=[0,2] 3(1856) minibatch=7 epoch=0 loss 5.000000e-01"
