"""`sc.tl.leiden` with scanpy's signature, running on libscanpy_b200 (B200, sm_100a).

Reference: src/scanpy/tools/_leiden.py:55-268, src/scanpy/tools/_utils_clustering.py:16-50,
src/scanpy/_utils/__init__.py:969-986.  The CUDA implementation (csrc/leiden.cu) optimises the same
objective both reference back-ends optimise for scanpy's defaults (RB configuration / modularity at
`resolution`), so `flavor` only selects which set of argument rules applies.
"""
from __future__ import annotations

from types import MappingProxyType
from typing import Any, Mapping, Sequence

import numpy as np
import pandas as pd

from . import _ops
from ._compat import LegacyRng, accepts_legacy_random_state, log_done, log_start, meta_random_state, seed_from_rng, warn


def _validate_flavor(flavor, *, partition_type, directed) -> str:
    """src/scanpy/tools/_leiden.py:231-268 (error texts pinned by tests/test_clustering.py:105-127)."""
    if flavor is None:
        flavor = "leidenalg"  # V1 preset default (src/scanpy/_settings/presets.py:271-277)
    if flavor == "igraph":
        if directed:
            raise ValueError("Cannot use igraph’s leiden implementation with a directed graph.")
        if partition_type is not None:
            raise ValueError("Do not pass in partition_type argument when using igraph.")
    elif flavor == "leidenalg":
        if partition_type is not None:
            raise NotImplementedError("custom `partition_type` is not implemented in scanpy_b200 "
                                      "(RBConfigurationVertexPartition / modularity only)")
    else:
        raise ValueError(f"flavor must be either 'igraph' or 'leidenalg', but {flavor!r} was passed.")
    return flavor


def _choose_graph(adata, obsp: str | None, neighbors_key: str | None):
    if obsp is not None and neighbors_key is not None:
        raise ValueError("You can't specify both obsp, neighbors_key. Please select only one.")
    if obsp is not None:
        return adata.obsp[obsp]
    key = "neighbors" if neighbors_key is None else neighbors_key
    if key not in adata.uns:
        if neighbors_key is None:
            raise ValueError("You need to run `pp.neighbors` first to compute a neighborhood graph.")
        raise KeyError(f"No {key!r} in .uns")
    conn_key = adata.uns[key].get("connectivities_key", "connectivities")
    if conn_key not in adata.obsp:
        raise ValueError("You need to run `pp.neighbors` first to compute a neighborhood graph.")
    return adata.obsp[conn_key]


def _restrict_adjacency(adata, restrict_key: str, *, restrict_categories: Sequence[str], adjacency):
    if not isinstance(restrict_categories[0], str):
        raise ValueError("You need to use strings to label categories, e.g. '1' instead of 1.")
    for c in restrict_categories:
        if c not in adata.obs[restrict_key].cat.categories:
            raise ValueError(f"{c!r} is not a valid category for {restrict_key!r}")
    restrict_indices = adata.obs[restrict_key].isin(restrict_categories).to_numpy()
    adjacency = adjacency[restrict_indices, :][:, restrict_indices]
    return adjacency, restrict_indices


def _rename_groups(adata, restrict_key, *, restrict_categories, restrict_indices, groups):
    all_groups = adata.obs[restrict_key].astype("U").copy()
    prefix = f"{'-'.join(restrict_categories)},"
    all_groups.iloc[np.flatnonzero(restrict_indices)] = [prefix + g for g in groups.astype("U")]
    return all_groups


@accepts_legacy_random_state(0)
def leiden(adata, resolution: float = 1, *, restrict_to=None, rng=None, key_added: str = "leiden", adjacency=None,
           directed: bool | None = None, use_weights: bool = True, n_iterations: int = -1, partition_type=None,
           neighbors_key: str | None = None, obsp: str | None = None, copy: bool = False, flavor: str | None = None,
           **clustering_args):
    """Leiden clustering (signature of `scanpy.tl.leiden`, tools/_leiden.py:55-72)."""
    _validate_flavor(flavor, partition_type=partition_type, directed=directed)
    if clustering_args:
        raise NotImplementedError(f"extra clustering_args {sorted(clustering_args)} are not implemented in scanpy_b200")
    meta_rs = meta_random_state(rng)
    start = log_start("running Leiden clustering")
    adata = adata.copy() if copy else adata
    if adjacency is None:
        adjacency = _choose_graph(adata, obsp, neighbors_key)
    restrict_indices = restrict_key = restrict_categories = None
    if restrict_to is not None:
        restrict_key, restrict_categories = restrict_to
        adjacency, restrict_indices = _restrict_adjacency(adata, restrict_key, restrict_categories=restrict_categories,
                                                          adjacency=adjacency)
    adj = adjacency.tocsr()
    if adj.dtype != np.float32:
        adj = adj.astype(np.float32)
    if not use_weights:
        adj = adj.copy()
        adj.data[:] = 1.0
    groups, modularity, _info = _ops.leiden(adj, resolution=1.0 if resolution is None else float(resolution),
                                            n_iterations=n_iterations, seed=seed_from_rng(rng))
    if restrict_to is not None:
        if key_added == "leiden":
            key_added += "_R"
        groups = _rename_groups(adata, restrict_key, restrict_categories=restrict_categories,
                                restrict_indices=restrict_indices, groups=groups)
        cats = sorted(map(str, np.unique(groups)), key=_natkey)
        adata.obs[key_added] = pd.Categorical(values=np.asarray(groups).astype("U"), categories=cats)
    else:
        # == pd.Categorical(values=groups.astype("U"), categories=natsorted(map(str, np.unique(groups))))
        # (_leiden.py:210-213): labels are 0..N-1 with no gaps, natsort == numeric order, so the codes are
        # the labels themselves; from_codes avoids materialising 1.3M Python strings
        n_groups = int(groups.max()) + 1 if len(groups) else 0
        cats = [str(c) for c in range(n_groups)]
        adata.obs[key_added] = pd.Categorical.from_codes(groups.astype(np.int32), categories=cats)
    adata.uns[key_added] = {}
    adata.uns[key_added]["params"] = dict(resolution=resolution, n_iterations=n_iterations, **meta_rs)
    adata.uns[key_added]["modularity"] = modularity
    log_done(start, f"found {len(cats)} clusters and added {key_added!r}, the cluster labels (adata.obs, categorical)")
    return adata if copy else None


def louvain(adata, resolution: float | None = None, *, random_state=0, restrict_to=None, key_added: str = "louvain",
            adjacency=None, flavor: str = "vtraag", directed: bool = True, use_weights: bool = False, partition_type=None,
            partition_kwargs: Mapping[str, Any] = MappingProxyType({}), neighbors_key: str | None = None,
            obsp: str | None = None, copy: bool = False):
    """Louvain clustering (signature of `scanpy.tl.louvain`, tools/_louvain.py:49-213).

    Both reference flavors maximise (RB-configuration) modularity by local moving + aggregation; the device kernel
    (sb2_louvain_csr_f32) optimises that objective on the SYMMETRIC graph: `directed=True` (the vtraag default) only
    changes how the reference counts the two arcs of each symmetric pair, which for a symmetric adjacency is the same
    objective up to the factor 2 in the edge total.  flavor='igraph' ignores `resolution` like the reference."""
    if flavor not in ("vtraag", "igraph"):
        if flavor == "taynaud":
            raise NotImplementedError("flavor='taynaud' (deprecated python-louvain) is not implemented in scanpy_b200")
        raise ValueError('`flavor` needs to be "vtraag" or "igraph" or "taynaud".')
    if flavor != "vtraag" and partition_type is not None:
        raise ValueError('`partition_type` is only a valid argument when `flavour` is "vtraag"')
    if partition_type is not None or dict(partition_kwargs):
        raise NotImplementedError("custom `partition_type` / `partition_kwargs` are not implemented in scanpy_b200 "
                                  "(RBConfigurationVertexPartition only)")
    start = log_start("running Louvain clustering")
    adata = adata.copy() if copy else adata
    if adjacency is None:
        adjacency = _choose_graph(adata, obsp, neighbors_key)
    restrict_indices = restrict_key = restrict_categories = None
    if restrict_to is not None:
        restrict_key, restrict_categories = restrict_to
        adjacency, restrict_indices = _restrict_adjacency(adata, restrict_key, restrict_categories=restrict_categories,
                                                          adjacency=adjacency)
    if flavor == "igraph" and resolution is not None:
        warn('`resolution` parameter has no effect for flavor "igraph"')
    adj = adjacency.tocsr()
    if adj.dtype != np.float32:
        adj = adj.astype(np.float32)
    if not use_weights:
        adj = adj.copy()
        adj.data[:] = 1.0
    gamma = 1.0 if (resolution is None or flavor == "igraph") else float(resolution)
    # `random_state` is the legacy form here (int | None | RandomState, _louvain.py:53): fold it to the kernels' integer seed
    seed = int(random_state) if isinstance(random_state, (int, np.integer)) else seed_from_rng(LegacyRng(random_state))
    groups, _q, _info = _ops.louvain(adj, resolution=gamma, seed=seed)
    if restrict_to is not None:
        if key_added == "louvain":
            key_added += "_R"
        groups = _rename_groups(adata, restrict_key, restrict_categories=restrict_categories,
                                restrict_indices=restrict_indices, groups=groups)
        cats = sorted(map(str, np.unique(groups)), key=_natkey)
        adata.obs[key_added] = pd.Categorical(values=np.asarray(groups).astype("U"), categories=cats)
    else:
        n_groups = int(groups.max()) + 1 if len(groups) else 0
        cats = [str(c) for c in range(n_groups)]
        adata.obs[key_added] = pd.Categorical.from_codes(groups.astype(np.int32), categories=cats)
    adata.uns[key_added] = {}
    adata.uns[key_added]["params"] = dict(resolution=resolution, random_state=random_state)
    log_done(start, f"found {len(cats)} clusters and added {key_added!r}, the cluster labels (adata.obs, categorical)")
    return adata if copy else None


def _natkey(s: str):
    import re

    return [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", s)]


from ._graph_tools import diffmap, paga, umap  # noqa: E402,F401  (SURVEY.md 8f rows f1, f3)
from ._rank_genes import rank_genes_groups  # noqa: E402,F401
