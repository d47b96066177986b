"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

Dev-time script (needs /root/reference; the GPU box does not have it, which is why the outputs are
committed).  It imports R: models/models.py and R: SimGFAToolbox/{dense,sparse}.py through the
third-party shims of `oracle/shims.py`, feeds them seeded synthetic inputs and stores inputs,
parameters, outputs and parameter gradients.

    python oracle/make_golden.py            # rewrites tests/golden/*.pt
"""
import hashlib
import importlib.util
import io
import contextlib
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("SNG_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)

from oracle import shims  # noqa: E402
from sngnn_b200 import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def load_reference_models():
    shims.install()
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import models.models as R  # the reference's own file, unmodified
    return R


def load_reference_file(rel, name):
    shims.install()
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def small_graph(N, Fd, E, C, seed, kind="clustered", symmetric=False, isolate=3):
    x = synth.make_features(N, Fd, kind, seed=seed, dup_frac=0.05, zero_rows=2 if N >= 32 else 0)
    ei = synth.make_graph(N, E, seed=seed + 1, symmetric=symmetric, hub_offset=4.0)
    if isolate:  # make the last `isolate` nodes isolated (empty scatter_max groups / trailing rows)
        keep = (ei[0] < N - isolate) & (ei[1] < N - isolate)
        ei = ei[:, keep]
    y = synth.make_labels(N, C, seed=seed + 2)
    return x, ei, y


def run_model(R, kind, x, ei, y, cfg, seed):
    N, Fd = x.shape
    C = int(y.max()) + 1
    torch.manual_seed(seed)
    if kind == "SNGNN":
        m = R.SNGNN(Fd, cfg["hidden"], C, cfg["layers"], bn=cfg.get("bn", False))
    elif kind == "SNGNN_Plus":
        m = R.SNGNN_Plus(Fd, cfg["hidden"], C, N, cfg["layers"], cfg["top_k"], cfg["thr"],
                         cfg["rsl"], 0.0, bn=cfg.get("bn", False))
    else:
        m = R.SNGNN_Plus_Plus(Fd, cfg["hidden"], C, N, cfg["layers"], cfg["top_k"], cfg["thr"], cfg["beta"],
                              cfg["rsl"], 0.0, bn=cfg.get("bn", False))
    if kind == "SNGNN":
        m.dropout = torch.nn.Dropout(0.0)  # R hard-codes p=0.5 (models.py:283); goldens are dropout-free
    m.train()
    data = synth.GraphData(x, ei)
    mask = torch.arange(N) % 2 == 0
    out = m(data)
    loss = F.nll_loss(out[mask], y[mask])
    loss.backward()
    grads = {k: p.grad.clone() for k, p in m.named_parameters()}
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return dict(kind=kind, cfg=cfg, state_dict=sd, logp=out.detach().clone(), loss=loss.detach().clone(), grads=grads)


def compact_run(run, seed, max_full=65536, stride=4):
    """A run that stays under 1 MB at the Chameleon shape: the initial parameters are the default initialisation under
    torch.manual_seed(seed), so only their SHA-256 is kept (tests/conftest.py:golden_state_dict regenerates and checks
    them); a gradient of more than `max_full` entries keeps every `stride`-th entry of the flattened tensor and the
    largest magnitude of the whole tensor (the scale of the relative error the tests take)."""
    init = dict(seed=seed, sha256={k: hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() for k, v in run["state_dict"].items()})
    grads = {k: g if g.numel() <= max_full else dict(stride=stride, values=g.reshape(-1)[::stride].clone(), absmax=g.abs().max())
             for k, g in run["grads"].items()}
    out = {k: v for k, v in run.items() if k != "state_dict"}
    return dict(out, init=init, grads=grads)


def main():
    os.makedirs(GOLD, exist_ok=True)
    R = load_reference_models()

    # ---- case A: tiny graph, every model / flag combination -----------------------------------
    x, ei, y = small_graph(64, 16, 320, 4, seed=10)
    runs = []
    for layers in (1, 2):
        runs.append(run_model(R, "SNGNN", x, ei, y, dict(hidden=8, layers=layers), seed=3))
        for rsl in (1, 0):
            for (k, thr) in ((1, 0.5), (3, 0.0), (10, 0.9), (4, -1.0)):
                cfg = dict(hidden=8, layers=layers, top_k=k, thr=thr, rsl=rsl)
                runs.append(run_model(R, "SNGNN_Plus", x, ei, y, cfg, seed=4))
                for beta in (0.0, 0.3):
                    runs.append(run_model(R, "SNGNN_Plus_Plus", x, ei, y, dict(cfg, beta=beta), seed=5))
    runs.append(run_model(R, "SNGNN_Plus_Plus", x, ei, y,
                          dict(hidden=8, layers=2, top_k=2, thr=0.1, rsl=1, beta=0.5, bn=True), seed=6))
    torch.save(dict(x=x, edge_index=ei.int(), y=y, runs=runs), os.path.join(GOLD, "models_tiny.pt"))
    print("models_tiny:", len(runs), "runs")

    # ---- case B: 1000 nodes, symmetric graph, hidden 32, 2 layers ------------------------------
    x, ei, y = small_graph(1000, 48, 8000, 5, seed=20, symmetric=True, isolate=5)
    runs = [
        run_model(R, "SNGNN", x, ei, y, dict(hidden=32, layers=2), seed=7),
        run_model(R, "SNGNN_Plus", x, ei, y, dict(hidden=32, layers=2, top_k=10, thr=0.0, rsl=1), seed=8),
        run_model(R, "SNGNN_Plus_Plus", x, ei, y, dict(hidden=32, layers=2, top_k=10, thr=0.3, rsl=1, beta=0.5), seed=9),
        run_model(R, "SNGNN_Plus_Plus", x, ei, y, dict(hidden=32, layers=1, top_k=2, thr=0.0, rsl=0, beta=0.2), seed=9),
    ]
    torch.save(dict(x=x, edge_index=ei.int(), y=y, runs=runs), os.path.join(GOLD, "models_small.pt"))
    print("models_small:", len(runs), "runs")

    # ---- case C: BASELINE config 1 (README.md:63): Chameleon shape, SNGNN++ 1 layer k=10 thr=0.9 ---
    N, Fd, E, C = synth.SHAPES["chameleon"]
    x = synth.make_features(N, Fd, "binary", seed=30)
    ei = synth.make_graph(N, E, seed=31, symmetric=False, hub_offset=4.0)
    y = synth.make_labels(N, C, seed=32)
    runs = [
        compact_run(run_model(R, "SNGNN_Plus_Plus", x, ei, y, dict(hidden=32, layers=1, top_k=10, thr=0.9, rsl=1, beta=0.0), seed=3), 3),
        compact_run(run_model(R, "SNGNN_Plus_Plus", x, ei, y, dict(hidden=32, layers=2, top_k=10, thr=0.5, rsl=1, beta=0.5), seed=3), 3),
    ]
    assert max(N, Fd) < 2 ** 15
    nz = x.nonzero().short()  # keep the file small: the 0/1 feature matrix is stored as its non-zero coordinates
    torch.save(dict(x_shape=(N, Fd), x_nz=nz, edge_index=ei.short(), y=y, runs=runs), os.path.join(GOLD, "models_chameleon.pt"))
    print("models_chameleon:", len(runs), "runs")

    # ---- toolbox: dense.py / sparse.py -------------------------------------------------------
    dense = load_reference_file("SimGFAToolbox/dense.py", "ref_dense")
    sparse = load_reference_file("SimGFAToolbox/sparse.py", "ref_sparse")
    tbu = load_reference_file("SimGFAToolbox/utils.py", "ref_tbutils")
    dt = load_reference_file("utils/data_transform.py", "ref_dt")
    x, ei, y = small_graph(300, 24, 2400, 4, seed=40, isolate=4)
    x1200, _, y1200 = small_graph(1200, 24, 10, 3, seed=41, isolate=0)  # >1 block of 1000 for the *_parted paths
    out = dict(x=x, edge_index=ei.int(), y=y, x1200=x1200, y1200=y1200)
    with contextlib.redirect_stdout(io.StringIO()):
        out["node_large_parted"] = dense.node_similarity_dense_large_parted(x1200)[1]
        out["class_large_1200"] = dense.class_similarity_dense_large(x1200, y1200)
        out["linked_large"] = dense.linked_node_similarity_dense_large(x, ei)
        out["nbr_large"] = dense.neighborhood_similarity_dense_large(x, ei)
        out["class_large"] = dense.class_similarity_dense_large(x, y)
        out["node_small"] = dense.node_similarity_dense_small(x)
        out["linked_small"] = dense.linked_node_similarity_dense_small(x, ei)
        out["nbr_small"] = dense.neighborhood_similarity_dense_small(x, ei)
        out["class_small"] = dense.class_similarity_dense_small(x, y)
        adj = tbu.edge_index_to_sparse_csc_tensor(x, ei)
        out["sp_node"] = sparse.node_similarity_sparse(adj)
        out["sp_linked"] = sparse.linked_node_similarity_sparse(adj, ei)
        out["sp_nbr"] = sparse.neighborhood_similarity_sparse(adj, ei)
        out["sp_class"] = sparse.class_similarity_sparse(adj, y)
        xs = synth.make_features(300, 24, "clustered", seed=42, zero_rows=0)  # no zero rows: R has no eps here
        out["esw_x"] = xs
        out["esw"] = dt.edge_similarity_weight(xs, ei)
    torch.save(out, os.path.join(GOLD, "toolbox.pt"))
    print("toolbox: done")
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
