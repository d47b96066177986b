"""Trainer for the three SN models -- the caller on top of the hot path (SURVEY.md §8 row f4).

Mirrors R: train.py for the part that drives SNGNN / SNGNN_Plus / SNGNN_Plus_Plus: the same flags with the same defaults
(R: train.py:23-65), the same step functions (R: train.py:70-117), the same epoch = train step + validation forward + test
forward (R: train.py:135-138), the same stopping rule (patience on the validation LOSS, test accuracy reported at the best
validation loss, R: train.py:150-158) and the same model factory arguments (R: train.py:305-315).  The 17 other model
families, the logger, the yaml config file and the dataset downloaders of the reference are out of scope: `--dataset` names a
synthetic shape of `sngnn_b200.synth.SHAPES` or a `.pt` file holding `{x, edge_index, y[, train_mask, val_mask, test_mask]}`.

    python -m sngnn_b200.train --model SNGNN_Plus_Plus --dataset chameleon --num_layers 1 --hidden_channels 32 \
        --top_k 10 --thr 0.9 --init_beta 0.0 --is_remove_self_loops 1 --epochs 50          (R: README.md:63)

The loss goes through `functional.nll_loss(out, y, mask)` (one fused pass) instead of `F.nll_loss(out[mask], y[mask])`:
same value, no gathered copies of an [N, C] matrix.  Everything runs on the CUDA device; there is no CPU path.
"""
import argparse
import os
import random
import time

import torch

from . import functional as SF
from . import synth
from .models import SNGNN, SNGNN_Plus, SNGNN_Plus_Plus

MODELS = ("SNGNN", "SNGNN_Plus", "SNGNN_Plus_Plus")


def parse_args(argv=None):
    """The flags of R: train.py:23-65 that reach the SN models (names, types and defaults unchanged)."""
    p = argparse.ArgumentParser(description="Train a similarity-navigated graph neural network")
    p.add_argument("--dataset", type=str, default="chameleon", help="synthetic shape name or path of a .pt graph file")
    p.add_argument("--model", type=str, default="SNGNN_Plus_Plus", help="one of " + ", ".join(MODELS))
    p.add_argument("--seed", type=int, default=1234, help="random seed")
    p.add_argument("--epochs", type=int, default=1000, help="number of epochs to train.")
    p.add_argument("--patience", type=int, default=100, help="patience")
    p.add_argument("--lr", type=float, default=0.01, help="initial learning rate.")
    p.add_argument("--weight_decay", type=float, default=5e-4, help="weight decay")
    p.add_argument("--dropout", type=float, default=0.5, help="dropout rate")
    p.add_argument("--hidden_channels", type=int, default=16, help="num of hidden channels for model")
    p.add_argument("--num_layers", type=int, default=2, help="num of network layers for model")
    p.add_argument("--part_id", type=int, default=0, help="data split part")
    p.add_argument("--top_k", type=int, default=1, help="select top_k for V4")
    p.add_argument("--thr", type=float, default=0.5, help="threshold  for V4")
    p.add_argument("--init_beta", type=float, default=0.5, help="trade off")
    p.add_argument("--is_remove_self_loops", type=int, default=1, help="whether to remove self-loops, 1 True, 0 False")
    p.add_argument("--device", type=str, default="cuda", help="CUDA device the run lives on")
    p.add_argument("--log-every", type=int, default=1, help="print every n-th epoch (0 = only the summary)")
    return p.parse_args(argv)


def set_random_seed(seed):
    """R: utils/seed.py:7-19."""
    random.seed(seed)
    os.environ["PYTHONHASHSEED"] = str(seed)
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed_all(seed)


def make_splits(num_nodes, part_id, device, fractions=(0.48, 0.32, 0.20)):
    """One of the fixed random train / validation / test partitions (the Geom-GCN style 48/32/20 splits the reference's
    WebKB / Wikipedia datasets ship as ten columns and select with `--part_id`, R: train.py:405-407)."""
    g = torch.Generator(device="cpu")
    g.manual_seed(10007 + int(part_id))
    perm = torch.randperm(num_nodes, generator=g)
    n_tr, n_va = int(fractions[0] * num_nodes), int(fractions[1] * num_nodes)
    masks = []
    for lo, hi in ((0, n_tr), (n_tr, n_tr + n_va), (n_tr + n_va, num_nodes)):
        m = torch.zeros(num_nodes, dtype=torch.bool)
        m[perm[lo:hi]] = True
        masks.append(m.to(device))
    return masks


def load_data(name, part_id=0, device="cuda"):
    """GraphData with .x .edge_index .y .train_mask .val_mask .test_mask, plus the number of classes."""
    key = name.lower()
    if key in synth.SHAPES:
        data, num_classes = synth.make_dataset(key, device=device)
    elif os.path.exists(name):
        blob = torch.load(name, map_location="cpu")
        data = synth.GraphData(blob["x"].float().to(device), blob["edge_index"].long().to(device), blob["y"].long().to(device))
        num_classes = int(blob.get("num_classes", int(data.y.max()) + 1))
        for k in ("train_mask", "val_mask", "test_mask"):
            if k in blob:
                m = blob[k]
                if m.dim() == 2:                                  # ten split columns, as the reference datasets carry them
                    m = m[:, part_id] if m.size(0) == data.x.size(0) else m[part_id]
                setattr(data, k, m.bool().to(device))
    else:
        raise ValueError(f"wrong dataset settings: {name!r} is neither one of {sorted(synth.SHAPES)} nor a file")
    if not hasattr(data, "train_mask"):
        data.train_mask, data.val_mask, data.test_mask = make_splits(data.x.size(0), part_id, device)
    return data, num_classes


def build_model(cfg, num_features, num_classes, num_nodes):
    """R: train.py:302-315 (argument order is the reference's)."""
    if cfg["model"] == "SNGNN":
        return SNGNN(num_features, cfg["hidden_channels"], num_classes, cfg["num_layers"])
    if cfg["model"] == "SNGNN_Plus":
        return SNGNN_Plus(num_features, cfg["hidden_channels"], num_classes, num_nodes, cfg["num_layers"], cfg["top_k"],
                          cfg["thr"], cfg["is_remove_self_loops"], cfg["dropout"])
    if cfg["model"] == "SNGNN_Plus_Plus":
        return SNGNN_Plus_Plus(num_features, cfg["hidden_channels"], num_classes, num_nodes, cfg["num_layers"], cfg["top_k"],
                               cfg["thr"], cfg["init_beta"], cfg["is_remove_self_loops"], cfg["dropout"])
    raise ValueError(f"wrong model settings: {cfg['model']!r} (this framework carries {', '.join(MODELS)})")


def _accuracy(output, y, mask):
    pred = output.max(dim=1)[1]
    return int((pred.eq(y) & mask).sum().item()) / max(int(mask.sum()), 1)


def train_step(model, data, optimizer):
    """R: train.py:70-85."""
    model.train()
    optimizer.zero_grad()
    output = model(data)
    train_loss = SF.nll_loss(output, data.y, data.train_mask)
    train_acc = _accuracy(output, data.y, data.train_mask)
    train_loss.backward()
    optimizer.step()
    return train_loss, train_acc


def _eval_step(model, data, mask):
    model.eval()
    with torch.no_grad():
        output = model(data)
        return SF.nll_loss(output, data.y, mask), _accuracy(output, data.y, mask)


def validate_step(model, data):
    """R: train.py:88-101."""
    return _eval_step(model, data, data.val_mask)


def test_step(model, data):
    """R: train.py:104-117."""
    return _eval_step(model, data, data.test_mask)


def train(model, data, optimizer, cfg, log=print):
    """R: train.py:120-160: stops after `patience` epochs without a new smallest validation loss; returns the test accuracy
    at that smallest validation loss (and the per-epoch history)."""
    dur, history = [], []
    final_test_acc, smallest_val_loss, curr_step = 0, float("inf"), 0
    for epoch in range(cfg["epochs"]):
        if data.x.is_cuda:
            torch.cuda.synchronize(data.x.device)
        t0 = time.time()
        train_loss, train_acc = train_step(model, data, optimizer)
        val_loss, val_acc = validate_step(model, data)
        test_loss, test_acc = test_step(model, data)
        train_loss, val_loss, test_loss = float(train_loss), float(val_loss), float(test_loss)     # device -> host: ends the epoch
        dur.append(time.time() - t0)
        history.append((train_loss, train_acc, val_loss, val_acc, test_loss, test_acc))
        if cfg.get("log_every", 1) and epoch % cfg["log_every"] == 0:
            log("Epoch: {:d} | Train_loss: {:.4f}, Train_acc:{:.4f}, Val_loss: {:.4f}, Val_acc:{:.4f}, Test_loss: {:.4f}, "
                "Test_acc:{:.4f}, Time(s): {:.4f}".format(epoch, train_loss, train_acc, val_loss, val_acc, test_loss, test_acc,
                                                          sum(dur) / len(dur)))
        if val_loss < smallest_val_loss:
            smallest_val_loss, final_test_acc, curr_step = val_loss, test_acc, 0
        else:
            curr_step += 1
        if curr_step == cfg["patience"]:
            break
    return final_test_acc, history


class ShardedData:
    """This rank's part of a dataset for the row-sharded trainer: rows [lo, hi) of x, y and the three masks, the whole edge_index,
    and the global mask counts (every rank loads the whole dataset, so they are known before training starts)."""

    def __init__(self, data, n, lo, hi):
        self.n, self.lo, self.hi = n, lo, hi
        self.x, self.edge_index, self.y = data.x[lo:hi].contiguous(), data.edge_index, data.y[lo:hi]
        self.masks, self.counts = {}, {}
        for k in ("train", "val", "test"):
            m = getattr(data, k + "_mask")
            self.masks[k] = m[lo:hi]
            self.counts[k] = int(m.sum())
        self.local_counts = {k: int(m.sum()) for k, m in self.masks.items()}


def _sharded_pass(sd, split, forward, loss_fn):
    """(loss term, local loss sum, local correct count) of one split on this rank's rows.  The loss term is the local masked
    mean times local / global count, so the terms of all ranks add up to the global masked mean; a rank without rows of the
    split contributes an exact 0 that still carries a gradient, because the backward runs collectives on every rank."""
    out = forward()
    mask, cnt = sd.masks[split], sd.local_counts[split]
    correct = (out.max(dim=1)[1].eq(sd.y) & mask).sum()
    if cnt == 0:
        return out.sum() * 0.0, out.new_zeros((), dtype=torch.float64), correct
    local = loss_fn(out, sd.y, mask)
    return local * (cnt / max(sd.counts[split], 1)), local.detach().double() * cnt, correct


def train_sharded(model, sd, optimizer, cfg, log=print, dropout=None, agg=None, fuse=None, bn_ops=None, loss_fn=None):
    """The epoch loop of `train` on row shards (dist.sharded_forward): a training step with `dropout` (a dist.RowDropout), then
    allreduce_grads and the optimizer; a validation and a test forward in eval mode; ONE all-reduce of an FP64 vector of loss sums
    and correct counts -- the epoch's host synchronisation -- from which every rank takes the same history and the same stopping
    decision.  `log` = None on the ranks that do not print.  agg / fuse / bn_ops / loss_fn replace the CUDA paths (gloo tests)."""
    from . import dist as D
    loss_fn = SF.nll_loss if loss_fn is None else loss_fn
    fwd = lambda: D.sharded_forward(model, sd.x, sd.edge_index, sd.n, agg=agg, fuse=fuse, bn_ops=bn_ops, dropout=dropout)
    dur, history = [], []
    final_test_acc, smallest_val_loss, curr_step = 0, float("inf"), 0
    for epoch in range(cfg["epochs"]):
        if sd.x.is_cuda:
            torch.cuda.synchronize(sd.x.device)
        t0 = time.time()
        model.train()
        optimizer.zero_grad()
        term, tr_sum, tr_cor = _sharded_pass(sd, "train", fwd, loss_fn)
        term.backward()
        D.allreduce_grads(model.parameters())
        optimizer.step()
        model.eval()
        with torch.no_grad():
            _, va_sum, va_cor = _sharded_pass(sd, "val", fwd, loss_fn)
            _, te_sum, te_cor = _sharded_pass(sd, "test", fwd, loss_fn)
        stats = torch.stack([v.to(torch.float64) for v in (tr_sum, tr_cor, va_sum, va_cor, te_sum, te_cor)])
        stats = D._all_reduce_sums(stats).tolist()                             # device -> host: ends the epoch
        dur.append(time.time() - t0)
        cnt = [max(sd.counts[k], 1) for k in ("train", "val", "test")]
        train_loss, val_loss, test_loss = stats[0] / cnt[0], stats[2] / cnt[1], stats[4] / cnt[2]
        train_acc, val_acc, test_acc = int(stats[1]) / cnt[0], int(stats[3]) / cnt[1], int(stats[5]) / cnt[2]
        history.append((train_loss, train_acc, val_loss, val_acc, test_loss, test_acc))
        if log is not None and cfg.get("log_every", 1) and epoch % cfg["log_every"] == 0:
            log("Epoch: {:d} | Train_loss: {:.4f}, Train_acc:{:.4f}, Val_loss: {:.4f}, Val_acc:{:.4f}, Test_loss: {:.4f}, "
                "Test_acc:{:.4f}, Time(s): {:.4f}".format(epoch, train_loss, train_acc, val_loss, val_acc, test_loss, test_acc,
                                                          sum(dur) / len(dur)))
        if val_loss < smallest_val_loss:
            smallest_val_loss, final_test_acc, curr_step = val_loss, test_acc, 0
        else:
            curr_step += 1
        if curr_step == cfg["patience"]:
            break
    return final_test_acc, history


def broadcast_parameters(model, src=0):
    """Make every rank's parameters and buffers rank `src`'s (w.weight lives in transposed storage: broadcast a contiguous copy)."""
    import torch.distributed as dist
    for t in list(model.parameters()) + list(model.buffers()):
        buf = t.data if t.data.is_contiguous() else t.data.contiguous()
        dist.broadcast(buf, src)
        if buf is not t.data:
            t.data.copy_(buf)


def main_sharded(cfg, log=print):
    """One rank of a torchrun launch (WORLD_SIZE, RANK, LOCAL_RANK set): NCCL on cuda:LOCAL_RANK, rows [lo, hi) of every node-level
    tensor, rank 0's initial parameters, train_sharded with a RowDropout seeded from --seed.  Every rank returns the same
    (final test accuracy, history); rank 0 logs."""
    import torch.distributed as dist
    from . import dist as D
    if not torch.cuda.is_available():
        raise RuntimeError("sngnn_b200.train needs a CUDA device (there is no CPU path)")
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    asked = torch.device(cfg["device"])
    if asked.type != "cuda" or (asked.index is not None and asked.index != device.index):
        raise ValueError(f"--device {cfg['device']} contradicts LOCAL_RANK={device.index}: under torchrun each rank runs on cuda:LOCAL_RANK")
    torch.cuda.set_device(device)
    dist.init_process_group("nccl", device_id=device)
    try:
        ws, rank = D.world()
        say = log if rank == 0 else (lambda *_: None)
        set_random_seed(cfg["seed"])
        cfg = dict(cfg, world_size=ws)
        say(f"Config:\n{cfg}")
        data, num_classes = load_data(cfg["dataset"], cfg["part_id"], device)
        n = data.x.size(0)
        say("train dataset len:{}, val dataset len:{}, test dataset len:{}".format(int(data.train_mask.sum()), int(data.val_mask.sum()),
                                                                                   int(data.test_mask.sum())))
        model = build_model(cfg, data.x.size(1), num_classes, n).to(device)
        broadcast_parameters(model)
        sd = ShardedData(data, n, *D.shard_bounds(n, ws, rank))
        del data
        optimizer = torch.optim.Adam(model.parameters(), lr=cfg["lr"], weight_decay=cfg["weight_decay"])
        say("number of epoch: {}".format(cfg["epochs"]))
        final_test_acc, history = train_sharded(model, sd, optimizer, cfg, log if rank == 0 else None, dropout=D.RowDropout(cfg["seed"]))
        say("Part {} final test acc: {:.4f}".format(cfg["part_id"], final_test_acc))
        return final_test_acc, history
    finally:
        dist.destroy_process_group()


def main(argv=None, log=print):
    """Single-GPU training; under torchrun (WORLD_SIZE set, 1 included) the row-sharded trainer, one rank per GPU."""
    args = parse_args(argv)
    cfg = dict(vars(args))
    if "WORLD_SIZE" in os.environ:
        return main_sharded(cfg, log)
    if not torch.cuda.is_available():
        raise RuntimeError("sngnn_b200.train needs a CUDA device (there is no CPU path)")
    device = torch.device(cfg["device"])
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    torch.cuda.set_device(device)
    set_random_seed(cfg["seed"])
    log(f"Config:\n{cfg}")
    data, num_classes = load_data(cfg["dataset"], cfg["part_id"], device)
    n = data.x.size(0)
    log("train dataset len:{}, val dataset len:{}, test dataset len:{}".format(int(data.train_mask.sum()), int(data.val_mask.sum()),
                                                                               int(data.test_mask.sum())))
    model = build_model(cfg, data.x.size(1), num_classes, n).to(device)
    optimizer = torch.optim.Adam(model.parameters(), lr=cfg["lr"], weight_decay=cfg["weight_decay"])
    log("number of epoch: {}".format(cfg["epochs"]))
    final_test_acc, history = train(model, data, optimizer, cfg, log)
    log("Part {} final test acc: {:.4f}".format(cfg["part_id"], final_test_acc))
    return final_test_acc, history


if __name__ == "__main__":
    main()
