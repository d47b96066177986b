import hashlib
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def golden_inputs(g):
    """(x, edge_index int64, y) of a models_*.pt file (chameleon stores x as non-zero coordinates)."""
    if "x" in g:
        x = g["x"]
    else:
        x = torch.zeros(g["x_shape"])
        nz = g["x_nz"].long()
        x[nz[:, 0], nz[:, 1]] = 1.0
    return x, g["edge_index"].long(), g["y"]


def golden_state_dict(g, run):
    """Initial parameters of a run of a models_*.pt file.  A run that records only `init` (oracle/make_golden.py:compact_run)
    started from the reference's default initialisation under torch.manual_seed(seed): each SNConv_plus_plus builds w, then
    lin, and resets lin and w; the model then resets every layer once more.  Regenerated here and checked against the
    recorded SHA-256 of every tensor."""
    if "state_dict" in run:
        return run["state_dict"]
    cfg, init = run["cfg"], run["init"]
    assert run["kind"] == "SNGNN_Plus_Plus" and not cfg.get("bn"), run["kind"]
    n, fd = g["x_shape"]
    dims = [fd] + [cfg["hidden"]] * (cfg["layers"] - 1) + [int(g["y"].max()) + 1]
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(init["seed"])
        layers = []
        for i, o in zip(dims[:-1], dims[1:]):
            w, lin = torch.nn.Linear(n, o), torch.nn.Linear(i, o)
            lin.reset_parameters()
            w.reset_parameters()
            layers.append((lin, w))
        for lin, w in layers:
            lin.reset_parameters()
            w.reset_parameters()
    sd = {}
    for l, (lin, w) in enumerate(layers):
        sd.update({f"lins.{l}.beta": torch.full((1,), float(cfg["beta"])), f"lins.{l}.w.weight": w.weight.detach(),
                   f"lins.{l}.w.bias": w.bias.detach(), f"lins.{l}.lin.weight": lin.weight.detach(), f"lins.{l}.lin.bias": lin.bias.detach()})
    assert sorted(sd) == sorted(init["sha256"])
    for k, v in sd.items():
        assert hashlib.sha256(v.numpy().tobytes()).hexdigest() == init["sha256"][k], f"regenerated initial {k} differs from the golden run's"
    return sd


def golden_grad(got, ref):
    """(got, ref, scale) for one parameter gradient of a golden run; a large gradient is stored as every `stride`-th entry of the
    flattened tensor plus the largest magnitude of the whole tensor."""
    if isinstance(ref, torch.Tensor):
        return got, ref, ref.abs().max()
    return got.reshape(-1)[::ref["stride"]], ref["values"], ref["absmax"]
