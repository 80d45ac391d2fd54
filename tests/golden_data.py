"""Stored outputs of the original implementation (``simple_models.py``, ``simple_utils.py``, ``lbfgsnew.py`` of the
upstream federated-pytorch-test scripts) for the tests that check this package against it.

Each such test module defines ``golden(ref)``: the reference side of its comparisons, run on ``ref.models``,
``ref.utils`` and ``ref.lbfgs`` with the same seeded inputs and weights the test uses.  Its arrays are stored in
``tests/golden/<module>.npz``; large tensors as a digest (shape, a seeded sample of values, plain and weighted sums)
so that every file stays small.  To regenerate after changing a test's inputs::

    python tests/golden_data.py --reference-src <directory holding simple_models.py, simple_utils.py, lbfgsnew.py>
"""
from __future__ import annotations

import argparse
import functools
import hashlib
import importlib
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_DIR = os.path.join(HERE, "golden")
MODULES = ["test_models", "test_utils_flat", "test_engine", "test_lbfgs"]
SAMPLE = 1024          # values kept per digested tensor (all of them when the tensor is this small)


def randn(*shape, seed: int = 0) -> torch.Tensor:
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def fill_(net: torch.nn.Module, seed: int = 0) -> torch.nn.Module:
    """Overwrite every floating-point entry of ``net.state_dict()``, in order, with seeded values of the usual
    magnitudes (weights uniform in +-1/sqrt(fan_in), norm scales near 1, small biases, positive running variances),
    so that two implementations with the same state_dict layout get the same weights."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, t in net.state_dict().items():
            if not t.is_floating_point():
                continue
            u = torch.rand(tuple(t.shape), generator=g, dtype=torch.float64) * 2 - 1
            if name.endswith("running_var"):
                v = 1.0 + 0.5 * u
            elif name.endswith("running_mean"):
                v = 0.1 * u
            elif t.dim() >= 2:
                v = u / (t[0].numel() ** 0.5)
            elif name.endswith("weight"):
                v = 1.0 + 0.1 * u
            else:
                v = 0.1 * u
            t.copy_(v.to(t.dtype))
    return net


def digest(t: torch.Tensor, prefix: str, k: int = SAMPLE) -> dict:
    """Shape, up to ``k`` values at seeded positions, sum, sum of magnitudes and a sum weighted by seeded uniforms."""
    flat = t.detach().reshape(-1).cpu()
    v = flat.double()
    n = v.numel()
    w = torch.rand(n, generator=torch.Generator().manual_seed(n), dtype=torch.float64)
    return {prefix + "/shape": np.array(t.shape, dtype=np.int64), prefix + "/sample": flat[_sample_idx(n, k)].numpy(),
            prefix + "/sums": np.array([float(v.sum()), float(v.abs().sum()), float((w * v).sum())])}


def assert_matches(t: torch.Tensor, g: dict, prefix: str, rtol: float = 1.3e-6, atol: float = 1e-5) -> None:
    """``t`` against a stored digest, elementwise on the sample and on the sums (tolerances scaled to the length)."""
    assert tuple(t.shape) == tuple(int(s) for s in g[prefix + "/shape"]), (prefix, tuple(t.shape))
    mine = digest(t, prefix, len(g[prefix + "/sample"]))
    torch.testing.assert_close(torch.from_numpy(mine[prefix + "/sample"]), torch.from_numpy(g[prefix + "/sample"]),
                               rtol=rtol, atol=atol, msg=lambda m: "%s: %s" % (prefix, m))
    s, ref = mine[prefix + "/sums"], g[prefix + "/sums"]
    bound = rtol * ref[1] + atol * max(1, t.numel())
    assert abs(s[0] - ref[0]) <= bound and abs(s[2] - ref[2]) <= bound, (prefix, s, ref)


def sha256(t: torch.Tensor) -> str:
    """Bit pattern of a float32 tensor, for comparisons that must be exact."""
    return hashlib.sha256(t.detach().float().contiguous().cpu().numpy().tobytes()).hexdigest()


@functools.lru_cache(maxsize=None)
def load(module: str) -> dict:
    with np.load(os.path.join(GOLDEN_DIR, module + ".npz"), allow_pickle=False) as f:
        return {k: f[k] for k in f.files}


def _sample_idx(n: int, k: int) -> torch.Tensor:
    if n <= k:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(n + 1))[:k].sort().values


def _import_file(path: str, name: str):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reference-src", required=True)
    args = ap.parse_args()
    sys.path.insert(0, os.path.dirname(HERE))
    ref = types.SimpleNamespace(**{k: _import_file(os.path.join(args.reference_src, f + ".py"), "_ref_" + f)
                                   for k, f in (("models", "simple_models"), ("utils", "simple_utils"), ("lbfgs", "lbfgsnew"))})
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    for name in MODULES:
        arrays = importlib.import_module(name).golden(ref)
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **arrays)
        print("%s: %d arrays, %d bytes" % (os.path.relpath(path, os.path.dirname(HERE)), len(arrays), os.path.getsize(path)))


if __name__ == "__main__":
    main()
