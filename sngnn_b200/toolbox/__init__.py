"""Sim-GFA toolbox on the B200 kernels: same function names as R: SimGFAToolbox/__init__.py:9-14.

Outputs follow the reference function by function, quirks included (SURVEY.md Appendix A.9).  Inputs may live on the
host or on the GPU; compute is always on the GPU (no CPU path), results come back on the input's device.
Plotting (R: SimGFAToolbox/plot.py) is presentation and out of scope: the two plot names raise NotImplementedError."""
from .dense import (node_similarity_dense_small, node_similarity_dense_large_parted, class_similarity_dense_small,
                    class_similarity_dense_large, linked_node_similarity_dense_large, linked_node_similarity_dense_small,
                    neighborhood_similarity_dense_large, neighborhood_similarity_dense_small, cosine_similarity_dense_small,
                    cosine_similarity, edge_similarity_weight, node_similarity_histogram)
from . import sharded  # noqa: F401  (row-sharded forms: one all-reduce of the class sums)
from .sparse import (cosine_similarity_sparse, class_similarity_sparse, neighborhood_similarity_sparse, node_similarity_sparse,
                     linked_node_similarity_sparse, edge_index_to_sparse_csc_tensor)


def plot_similarity_distribution(*a, **k):
    raise NotImplementedError("plotting is out of scope of the hot path (R: SimGFAToolbox/plot.py)")


def plot_class_similarity(*a, **k):
    raise NotImplementedError("plotting is out of scope of the hot path (R: SimGFAToolbox/plot.py)")


__all__ = ['cosine_similarity_sparse', 'node_similarity_sparse', 'linked_node_similarity_sparse', 'class_similarity_sparse',
           'plot_class_similarity', 'plot_similarity_distribution', 'edge_index_to_sparse_csc_tensor',
           'node_similarity_dense_small', 'node_similarity_dense_large_parted', 'class_similarity_dense_small',
           'class_similarity_dense_large', 'linked_node_similarity_dense_large', 'linked_node_similarity_dense_small',
           'neighborhood_similarity_dense_large', 'neighborhood_similarity_dense_small']
