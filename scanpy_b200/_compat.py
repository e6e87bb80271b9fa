"""Small host-side pieces of scanpy's runtime that the three hot-path functions lean on.

* `MiniAnnData` — a duck-typed stand-in for `anndata.AnnData` (anndata is not installed in the build
  image).  The public functions only use `.X .obs .var .var_names .obsm .varm .obsp .uns .layers .raw
  .n_obs .n_vars .shape .is_view .copy()` and `adata[:, mask]`, so a real AnnData works unchanged.
* `settings` — the two constants the path reads (`N_PCS`, `n_jobs`; src/scanpy/_settings/__init__.py:83,132)
  plus verbosity-free logging with the reference's message texts (src/scanpy/logging.py:100-131).
* `accepts_legacy_random_state` — the `random_state=` <-> `rng=` shim of
  src/scanpy/_utils/random.py:182-208: a bare call or `random_state=` records
  `params['random_state']` in `.uns`, an explicit `rng=` does not.
"""
from __future__ import annotations

import logging
import time
import warnings
from functools import wraps
from types import SimpleNamespace

import numpy as np
import pandas as pd
from scipy import sparse

logger = logging.getLogger("scanpy_b200")

settings = SimpleNamespace(N_PCS=50, n_jobs=4, chunk_size=50_000)  # anndata's default chunk_size for chunked_X is 6000; the device path prefers larger row chunks


def log_start(msg: str) -> float:
    logger.info(msg)
    return time.perf_counter()


def log_done(start: float, deep: str = "") -> None:
    logger.info("    finished (%.3fs)%s", time.perf_counter() - start, (" " + deep) if deep else "")


def warn(msg: str, category=UserWarning) -> None:
    warnings.warn(msg, category, stacklevel=3)


class LegacyRng:
    """Marker: the caller used the legacy `random_state` form (value kept in `.arg`)."""

    def __init__(self, arg):
        self.arg = arg

    def generator(self) -> np.random.Generator:
        return np.random.default_rng(self.arg if self.arg is not None else None)


def accepts_legacy_random_state(default_seed):
    """`f(..., rng=None)` gains a `random_state=` keyword; neither given -> legacy default seed."""

    def deco(fn):
        @wraps(fn)
        def wrapper(*args, random_state="__unset__", rng=None, **kw):
            if rng is not None and random_state != "__unset__":
                raise TypeError("Specify at most one of `rng` and `random_state`.")
            if rng is None:
                rng = LegacyRng(default_seed if random_state == "__unset__" else random_state)
            return fn(*args, rng=rng, **kw)

        return wrapper

    return deco


def seed_from_rng(rng) -> int:
    """Integer seed for the CUDA kernels from either form."""
    if isinstance(rng, LegacyRng):
        if isinstance(rng.arg, (int, np.integer)):
            return int(rng.arg) & 0xFFFFFFFFFFFFFFFF
        return int(np.random.default_rng(None if rng.arg is None else rng.arg).integers(0, 2**31 - 1))
    return int(np.random.default_rng(rng).integers(0, 2**31 - 1))


def meta_random_state(rng) -> dict:
    return dict(random_state=rng.arg) if isinstance(rng, LegacyRng) else {}


class _AxisArrays(dict):
    pass


class MiniAnnData:
    """Minimal AnnData look-alike: enough surface for pca/neighbors/leiden and their tests."""

    def __init__(self, X=None, obs=None, var=None, obsm=None, varm=None, obsp=None, uns=None):
        self.X = X
        n_obs, n_vars = X.shape
        self.obs = obs if obs is not None else pd.DataFrame(index=pd.RangeIndex(n_obs).astype(str))
        self.var = var if var is not None else pd.DataFrame(index=pd.RangeIndex(n_vars).astype(str))
        self.obsm = _AxisArrays(obsm or {})
        self.varm = _AxisArrays(varm or {})
        self.obsp = _AxisArrays(obsp or {})
        self.uns = dict(uns or {})
        self.layers = {}
        self.raw = None  # anything with .X and .var_names (e.g. another MiniAnnData), as `anndata.AnnData.raw`
        self.is_view = False
        self.isbacked = False

    @property
    def var_names(self) -> pd.Index:
        return self.var.index

    @property
    def shape(self):
        return self.X.shape

    @property
    def n_obs(self):
        return self.X.shape[0]

    @property
    def n_vars(self):
        return self.X.shape[1]

    def copy(self):
        import copy

        new = MiniAnnData(self.X.copy(), self.obs.copy(), self.var.copy(),
                          {k: v.copy() for k, v in self.obsm.items()}, {k: v.copy() for k, v in self.varm.items()},
                          {k: v.copy() for k, v in self.obsp.items()}, copy.deepcopy(self.uns))
        new.raw = self.raw.copy() if self.raw is not None else None
        return new

    def __getitem__(self, idx):
        if not (isinstance(idx, tuple) and len(idx) == 2 and isinstance(idx[0], slice) and idx[0] == slice(None)):
            raise NotImplementedError("MiniAnnData only supports adata[:, var_mask]")
        mask = np.asarray(idx[1])
        x = self.X[:, mask]
        sub = MiniAnnData(x, self.obs, self.var.loc[mask] if mask.dtype == bool else self.var.iloc[mask])
        sub.is_view = True
        return sub


def is_anndata_like(obj) -> bool:
    return all(hasattr(obj, a) for a in ("X", "obs", "var", "obsm", "varm", "obsp", "uns"))


def as_csr_f32(x):
    """Input matrix -> scipy CSR with float32 data (float64 is down-cast: the kernels compute in fp32
    storage / fp64 accumulation; dense input is converted)."""
    if sparse.issparse(x):
        x = x.tocsr()
    else:
        x = sparse.csr_matrix(np.asarray(x))
    if x.dtype != np.float32:
        x = x.astype(np.float32)
    if not x.has_canonical_format:
        x = x.copy()
        x.sum_duplicates()
    return x
