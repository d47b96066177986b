"""Drop-in modules for the reference's similarity-navigated models.

Same class names, constructor argument names / order / defaults (including the `droput_rate` spelling),
parameter names (`lins.{l}.lin.{weight,bias}`, `.w.{weight,bias}`, `.beta`, `.bias`, `bns.{l}.*`), forward
signature and outputs as R: models/models.py:35-334, so `train.py:305-315` can construct them unchanged and a
reference state_dict loads.  The work between `lin(x)` and the layer output runs in libsng.so.

Extra keyword-only options (not in the reference; defaults reproduce it):
  candidates  = 'edges'      neighbours are chosen among graph in-neighbours (what models.py does, SURVEY.md D1)
              | 'all_pairs'  neighbours are chosen among ALL nodes with the tensor-core kNN builder (north_star 1-2)
  denominator = 'candidates' mean divides by the size of the candidate list (PyG aggr='mean', SURVEY.md D3)
              | 'selected'   mean divides by the number of selected neighbours
"""
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn.parameter import Parameter

from . import _C
from . import functional as SF
from . import graph as G


def _as_bool(flag):
    # R: models/models.py:44-47 -- only the integer 1 (or True) enables removal
    return flag == 1


class _SNConvBase(nn.Module):
    @staticmethod
    def _check_width(out_channels):
        # the edge kernels are instantiated up to SNG_MAX_CHANNELS; fail at construction, not at the first forward
        if SF.padded_channels(out_channels) > _C.MAX_CHANNELS:
            raise ValueError(f"out_channels={out_channels}: the B200 edge kernels support at most {_C.MAX_CHANNELS} channels per "
                             "layer (the reference accepts any width)")

    def _init_bias(self, bias, out_channels):
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)

    def _zero_bias(self):
        if self.bias is not None:
            self.bias.data.fill_(0)

    def _hidden(self, x):
        cp = SF.padded_channels(self.lin.out_features)
        return SF.linear_padded(x, self.lin.weight, self.lin.bias, cp)

    def _hidden_norm(self, x):
        """(h, 1/||h||) -- R: models/models.py:121-122 -- in one pass over x when the shape allows (else inv_norm = None)."""
        return SF.lin_norm(x, self.lin.weight, self.lin.bias, SF.padded_channels(self.lin.out_features))


class SNConv(_SNConvBase):
    """R: models/models.py:305-334 -- cosine-weighted mean over all in-neighbours incl. a self loop."""

    def __init__(self, in_channels, out_channels, aggr="mean", bias: bool = True):
        super().__init__()
        if aggr != "mean":
            raise NotImplementedError("only aggr='mean' (the value every reference call site uses)")
        self._check_width(out_channels)
        self.lin = nn.Linear(in_channels, out_channels)
        self._init_bias(bias, out_channels)
        self.reset_parameters()

    def reset_parameters(self):
        self.lin.reset_parameters()
        self._zero_bias()

    def forward(self, x, edge_index):
        g = G.prepare(edge_index, x.size(0), remove_self_loops=False)
        h, inv = self._hidden_norm(x)
        out = SF.edge_topk_agg(h, g, None, None, inv_norm=inv)[:, :self.lin.out_features]
        if self.bias is not None:
            out = out + self.bias
        return out


class SNConv_plus(_SNConvBase):
    """R: models/models.py:214-263."""

    def __init__(self, in_channels, out_channels, num_nodes, top_k=2, thr=0.0, is_remove_self_loops=True,
                 bias: bool = False, aggr="mean", *, candidates="edges", denominator="candidates"):
        super().__init__()
        if aggr != "mean":
            raise NotImplementedError("only aggr='mean'")
        self.top_k, self.thr = top_k, thr
        self.num_nodes = num_nodes
        self.is_remove_self_loops = is_remove_self_loops
        self.candidates, self.denominator = candidates, denominator
        self._check_width(out_channels)
        self.lin = nn.Linear(in_channels, out_channels)
        self._init_bias(bias, out_channels)
        self.reset_parameters()

    def reset_parameters(self):
        self.lin.reset_parameters()
        self._zero_bias()

    def _check_options(self):
        if self.candidates not in ("edges", "all_pairs"):
            raise ValueError(f"candidates={self.candidates!r}")
        if self.denominator not in ("candidates", "selected"):
            raise ValueError(f"denominator={self.denominator!r}")

    def _aggregate(self, h, g, inv=None):
        """out_1 of R: models/models.py:239 / :132.  top_k <= 0: the reference runs zero scatter_max rounds, every weight
        stays 0 and out_1 = 0 (with zero -- not missing -- gradients)."""
        if self.top_k <= 0:
            return h * 0.0
        if self.candidates == "edges":
            return SF.edge_agg(h, g, self.top_k, self.thr, inv_norm=inv, denominator=self.denominator)
        from . import simknn
        return simknn.allpairs_topk_agg(h, self.top_k, self.thr, bool(self.is_remove_self_loops), self.denominator)

    def forward(self, x, edge_index):
        self._check_options()
        g = G.prepare(edge_index, x.size(0), remove_self_loops=bool(self.is_remove_self_loops))
        h, inv = self._hidden_norm(x)
        out = self._aggregate(h, g, inv)[:, :self.lin.out_features]
        if self.bias is not None:
            out = out + self.bias
        return out


class SNConv_plus_plus(SNConv_plus):
    """R: models/models.py:89-158 -- adds beta * (A @ W^T + b_w), beta learnable, initialised to init_beta."""

    def __init__(self, in_channels, out_channels, num_nodes, top_k=2, thr=0.0, init_beta=0.5, is_remove_self_loops=True,
                 bias: bool = False, aggr="mean", *, candidates="edges", denominator="candidates"):
        nn.Module.__init__(self)
        if aggr != "mean":
            raise NotImplementedError("only aggr='mean'")
        self.top_k, self.thr = top_k, thr
        self._check_width(out_channels)
        self.w = nn.Linear(num_nodes, out_channels)
        # w.weight keeps the reference's name and shape [C, N] but lives in TRANSPOSED storage ([N, C] row-major): the
        # kernels gather rows of W^T, the gradient comes out row by row, and Adam (state allocated with preserve_format)
        # then runs on the same layout -- no transpose copy of a 209 MB parameter (pokec, C = 32) anywhere in a step.
        self.w.weight = Parameter(torch.empty(num_nodes, out_channels).t())
        self.num_nodes = num_nodes
        self.is_remove_self_loops = is_remove_self_loops
        self.candidates, self.denominator = candidates, denominator
        self.lin = nn.Linear(in_channels, out_channels)
        self.beta = Parameter(torch.empty(1))
        self.init_beta = init_beta
        self._init_bias(bias, out_channels)
        self.reset_parameters()

    def reset_parameters(self):
        self.lin.reset_parameters()
        self._zero_bias()
        self.w.reset_parameters()
        self.beta.data.fill_(self.init_beta)

    def forward(self, x, edge_index):
        if x.size(0) != self.num_nodes:
            raise RuntimeError(f"SNConv_plus_plus was built for num_nodes={self.num_nodes} but got {x.size(0)} rows")
        self._check_options()
        g = G.prepare(edge_index, x.size(0), remove_self_loops=bool(self.is_remove_self_loops))
        h, inv = self._hidden_norm(x)
        if self.top_k > 0 and self.candidates == "edges" and g.symmetric:
            # in-lists == out-lists: the structural term rides on the aggregation's own pass over the edges (one kernel)
            out = SF.edge_agg(h, g, self.top_k, self.thr, structural=(self.w.weight, self.w.bias, self.beta, self.bias), inv_norm=inv,
                              denominator=self.denominator)
        else:
            out = SF.PPFuse.apply(self._aggregate(h, g, inv), self.w.weight, self.w.bias, self.beta, self.bias, g)
        return out[:, :self.lin.out_features]


class _SNStack(nn.Module):
    """Layer stack shared by the three models (R: models/models.py:76-86, 201-211, 293-303)."""

    def _build(self, make_conv, in_channels, hidden_channels, out_channels, num_layers, bn):
        self.bn = bn
        self.lins = nn.ModuleList()
        if self.bn:
            self.bns = nn.ModuleList()
        if num_layers == 1:
            self.lins.append(make_conv(in_channels, out_channels))
        else:
            self.lins.append(make_conv(in_channels, hidden_channels))
            if self.bn:
                self.bns.append(nn.BatchNorm1d(hidden_channels))
            for _ in range(num_layers - 2):
                self.lins.append(make_conv(hidden_channels, hidden_channels))
                if self.bn:
                    self.bns.append(nn.BatchNorm1d(hidden_channels))
            self.lins.append(make_conv(hidden_channels, out_channels))

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()
        if self.bn:
            for bn in self.bns:
                bn.reset_parameters()

    def forward(self, data):
        x, edge_index = data.x, data.edge_index
        for i, lin in enumerate(self.lins[:-1]):
            x = F.relu(lin(x, edge_index))
            if self.bn:
                x = self.bns[i](x)
            x = self.dropout(x)
        x = self.lins[-1](x, edge_index)
        return F.log_softmax(x, dim=1)


class SNGNN(_SNStack):
    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, bn=False):
        super().__init__()
        self._build(lambda i, o: SNConv(i, o), in_channels, hidden_channels, out_channels, num_layers, bn)
        self.dropout = nn.Dropout(p=0.5)            # fixed, R: models/models.py:283
        self.reset_parameters()


class SNGNN_Plus(_SNStack):
    def __init__(self, in_channels, hidden_channels, out_channels, num_nodes, num_layers, top_k=2, thr=0.0,
                 is_remove_self_loops=1, droput_rate=0.5, bn=False, *, candidates="edges", denominator="candidates"):
        super().__init__()
        self.top_k, self.thr, self.num_nodes = top_k, thr, num_nodes
        self.is_remove_self_loops = _as_bool(is_remove_self_loops)
        # the model's `bn` flag lands in the conv's `bias` slot (positional quirk of R: models/models.py:177-178)
        self._build(lambda i, o: SNConv_plus(i, o, num_nodes, top_k, thr, self.is_remove_self_loops, bn,
                                             candidates=candidates, denominator=denominator),
                    in_channels, hidden_channels, out_channels, num_layers, bn)
        self.dropout = nn.Dropout(p=droput_rate)
        self.reset_parameters()


class SNGNN_Plus_Plus(_SNStack):
    def __init__(self, in_channels, hidden_channels, out_channels, num_nodes, num_layers, top_k=2, thr=0.0,
                 init_beta=0.5, is_remove_self_loops=1, droput_rate=0.5, bn=False, *, candidates="edges",
                 denominator="candidates"):
        super().__init__()
        self.top_k, self.thr, self.init_beta, self.num_nodes = top_k, thr, init_beta, num_nodes
        self.is_remove_self_loops = _as_bool(is_remove_self_loops)
        self._build(lambda i, o: SNConv_plus_plus(i, o, num_nodes, top_k, thr, init_beta, self.is_remove_self_loops, bn,
                                                  candidates=candidates, denominator=denominator),
                    in_channels, hidden_channels, out_channels, num_layers, bn)
        self.dropout = nn.Dropout(p=droput_rate)
        self.reset_parameters()
