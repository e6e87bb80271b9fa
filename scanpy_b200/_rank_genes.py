"""`sc.tl.rank_genes_groups` with scanpy's signature (ScanpyV1 preset), the reductions on libscanpy_b200.

Reference: src/scanpy/tools/_rank_genes_groups.py:743-1029.  The device computes the grouped per-gene statistics
(sb2_rank_genes_group_stats) and the Wilcoxon rank sums / tie terms (sb2_rank_genes_wilcoxon); everything after that
works on [groups x genes] arrays on the host with the reference's formulas: the Chan leave-one-out rest variance
(:198-237), Welch's t-test (:454-503), the rank-sum z-scores (:505-579), the multiple-testing corrections and log fold
changes (:678-740), and the top-n selection (:42-49).

Float64 data is ranked after a cast to float32 (with a UserWarning); integer and float32 data are ranked exactly.
"""
from __future__ import annotations

import numpy as np
import pandas as pd
from scipy import sparse

from . import _abi, _ops
from ._compat import log_done, log_start, logger, warn

_METHODS = ("logreg", "t-test", "wilcoxon", "wilcoxon_illico", "t-test_overestim_var")
_NOT_IMPLEMENTED = ("logreg", "wilcoxon_illico")


def _select_top_n(scores: np.ndarray, n_top: int) -> np.ndarray:
    """src/scanpy/tools/_rank_genes_groups.py:42-49 (same calls, so tied scores order the same way)."""
    reference_indices = np.arange(scores.shape[0], dtype=int)
    partition = np.argpartition(scores, -n_top)[-n_top:]
    partial_indices = np.argsort(scores[partition])[::-1]
    return reference_indices[partition][partial_indices]


def _fdr_bh(pvals: np.ndarray) -> np.ndarray:
    """statsmodels' multipletests(method='fdr_bh') corrected p-values: sort, p * n / rank, reversed cumulative minimum,
    clip at 1, unsort."""
    order = np.argsort(pvals)
    p_sorted = pvals[order]
    n = p_sorted.shape[0]
    corrected = p_sorted / (np.arange(1, n + 1) / float(n))
    corrected = np.minimum.accumulate(corrected[::-1])[::-1]
    corrected[corrected > 1] = 1
    out = np.empty_like(corrected)
    out[order] = corrected
    return out


def _chan_combine(n_a, mean_a, m2_a, n_b, mean_b, m2_b):
    """scanpy.get._aggregated._chan_combine over arrays of genes (n_a, n_b scalars)."""
    if n_a == 0.0:
        return n_b, mean_b, m2_b
    if n_b == 0.0:
        return n_a, mean_a, m2_a
    n = n_a + n_b
    delta = mean_b - mean_a
    return n, (n_a * mean_a + n_b * mean_b) / n, m2_a + m2_b + delta * delta * n_a * n_b / n


def _vars_rest(group_counts: np.ndarray, mean: np.ndarray, m2: np.ndarray, k: int) -> np.ndarray:
    """Leave-one-out variance of every selected group's rest (:198-237), vectorised over genes."""
    n_groups = group_counts.shape[0]

    def scan(order):
        acc = [None] * n_groups
        state = (0.0, 0.0, 0.0)
        for i in order:
            state = _chan_combine(*state, float(group_counts[i]), mean[i], m2[i])
            acc[i] = state
        return acc

    upto = scan(range(n_groups))
    after = scan(range(n_groups - 1, -1, -1))
    out = np.zeros((k, mean.shape[1]))
    for g in range(k):
        n_b, _, m2_b = after[g + 1]
        if g >= 1:
            n_r, _, m2_r = _chan_combine(*upto[g - 1], *after[g + 1])
        else:
            n_r, m2_r = n_b, m2_b
        with np.errstate(divide="ignore", invalid="ignore"):
            out[g] = m2_r / (n_r - 1.0)
    return out


def _select_groups(col: pd.Series, groups_order_subset):
    """src/scanpy/_utils/__init__.py:798-841 -> (groups_order ndarray, masks bool [k, n])."""
    cats = col.cat.categories
    values = col.to_numpy()
    masks = np.zeros((len(cats), col.size), dtype=bool)
    arr = col.array
    for iname, name in enumerate(cats):
        masks[iname] = (name == values) if name in arr else (str(iname) == values)
    if isinstance(groups_order_subset, str) and groups_order_subset == "all":
        return cats.to_numpy(), masks
    ids = [np.flatnonzero(cats.array == name)[0] for name in groups_order_subset]
    if len(ids) == 0:
        ids = np.flatnonzero(np.isin(np.arange(len(cats)).astype(str), np.array(groups_order_subset)))
    if len(ids) == 0:
        raise RuntimeError(f"{np.array(groups_order_subset)} invalid! specify valid groups_order (or indices) from {cats}")
    return cats[ids].to_numpy(), masks[ids]


def _sanitize_obs(adata) -> None:
    """String columns of .obs -> categoricals (anndata's `_sanitize`, called by sanitize_anndata)."""
    for name in adata.obs.columns:
        c = adata.obs[name]
        if isinstance(c.dtype, pd.CategoricalDtype):
            continue
        if pd.api.types.is_string_dtype(c.dtype) and not pd.api.types.is_bool_dtype(c.dtype):
            adata.obs[name] = pd.Categorical(c)


def _as_ranked_csr(x) -> sparse.csr_matrix:
    """The matrix the kernels read: float32 CSR.  Float64 is cast (one warning), integers are exact below 2**24."""
    if type(x).__module__.startswith("dask"):
        raise NotImplementedError("rank_genes_groups on dask arrays is not implemented in scanpy_b200")
    if hasattr(x, "to_memory") or type(x).__name__.startswith(("Backed", "Dataset")):
        raise NotImplementedError("rank_genes_groups on backed (on-disk) matrices is not implemented in scanpy_b200")
    dtype = x.dtype
    if dtype == np.float64:
        warn("rank_genes_groups: float64 data is ranked after a cast to float32 (scanpy_b200 kernels read float32)",
             UserWarning)
    if sparse.issparse(x):
        x = x.tocsr()
    else:
        x = sparse.csr_matrix(np.asarray(x))
    if x.dtype != np.float32:
        x = x.astype(np.float32)
    return x


def _check_nonnegative_integers(x: sparse.csr_matrix) -> bool:
    data = x.data
    return not np.signbit(data).any() and not np.any((data % 1) != 0)


def rank_genes_groups(adata, groupby: str, *, mask_var=None, use_raw: bool | None = None, groups="all",
                      reference: str = "rest", n_genes: int | None = None, rankby_abs: bool = False, pts: bool = False,
                      key_added: str | None = None, copy: bool = False, method: str | None = "t-test",
                      corr_method: str = "benjamini-hochberg", tie_correct: bool = False, layer: str | None = None,
                      mean_in_log_space: bool = True, **kwds):
    """Rank genes for characterizing groups (signature and outputs of `scanpy.tl.rank_genes_groups`,
    tools/_rank_genes_groups.py:743-1029, ScanpyV1 preset: method='t-test', mean_in_log_space=True).

    Methods 't-test', 't-test_overestim_var' and 'wilcoxon' (optionally `tie_correct`) run on the device; 'logreg',
    'wilcoxon_illico', dask and backed matrices raise NotImplementedError.  At most 1024 groups are compared."""
    from .pp import _check_mask

    if method is None:
        method = "t-test"
    mask_var = _check_mask(adata, mask_var, "var")
    raw = getattr(adata, "raw", None)
    if use_raw is None:
        use_raw = raw is not None
    elif use_raw is True and raw is None:
        raise ValueError("Received `use_raw=True`, but `adata.raw` is empty.")
    if "only_positive" in kwds:
        rankby_abs = not kwds.pop("only_positive")  # backwards compat
    if method not in _METHODS:
        raise ValueError(f"Method must be one of {_METHODS}.")
    avail_corr = {"benjamini-hochberg", "bonferroni"}
    if corr_method not in avail_corr:
        raise ValueError(f"Correction method must be one of {avail_corr}.")
    if method in _NOT_IMPLEMENTED:
        raise NotImplementedError(f"method={method!r} is not implemented in scanpy_b200")
    start = log_start("ranking genes")

    adata = adata.copy() if copy else adata
    _sanitize_obs(adata)
    if isinstance(groups, str) and groups == "all":
        groups_order = "all"
    elif isinstance(groups, (str, int)):
        raise ValueError("Specify a sequence of groups")
    else:
        groups_order = list(groups)
        if isinstance(groups_order[0], int):
            groups_order = [str(n) for n in groups_order]
        if reference != "rest" and reference not in set(groups_order):
            groups_order += [reference]
    if reference != "rest" and reference not in adata.obs[groupby].cat.categories:
        cats = adata.obs[groupby].cat.categories.tolist()
        raise ValueError(f"reference = {reference} needs to be one of groupby = {cats}.")

    if key_added is None:
        key_added = "rank_genes_groups"
    adata.uns[key_added] = {}
    adata.uns[key_added]["params"] = dict(groupby=groupby, reference=reference, method=method, use_raw=use_raw,
                                          layer=layer, corr_method=corr_method)

    # --- _RankGenes.__init__ (:240-317)
    base = adata.uns.get("log1p", {}).get("base")
    log_scale = float(np.log(base)) if base is not None else 1.0
    expm1_func = (lambda v: np.expm1(v * np.log(base))) if base is not None else np.expm1
    col = adata.obs[groupby]
    groups_order, groups_masks_obs = _select_groups(col, groups_order)
    invalid = set(groups_order) & set(col.value_counts().loc[lambda c: c < 2].index)
    if invalid:
        raise ValueError(f"Could not calculate statistics for groups {', '.join(invalid)} "
                         "since they only contain one sample.")
    if layer is not None:
        if use_raw:
            raise ValueError("Cannot specify `layer` and have `use_raw=True`.")
        x, var_names = adata.layers[layer], adata.var_names
    elif use_raw and raw is not None:
        x, var_names = raw.X, raw.var_names
    else:
        x, var_names = adata.X, adata.var_names
    if getattr(adata, "isbacked", False) and layer is None and not use_raw:
        raise NotImplementedError("rank_genes_groups on backed (on-disk) matrices is not implemented in scanpy_b200")
    k = groups_masks_obs.shape[0]
    if k > _abi.RANK_GENES_MAX_GROUPS:
        raise NotImplementedError(f"rank_genes_groups compares at most {_abi.RANK_GENES_MAX_GROUPS} groups in "
                                  f"scanpy_b200 ({k} were selected)")
    x = _as_ranked_csr(x)
    if mask_var is not None:
        x = x[:, mask_var]
        var_names = var_names[mask_var]
    ireference = None if reference == "rest" else int(np.where(groups_order == reference)[0][0])

    if _check_nonnegative_integers(x):
        logger.warning("It seems you use rank_genes_groups on the raw count data. "
                       "Please logarithmize your data before calling rank_genes_groups.")
    n_genes_user = n_genes
    if n_genes_user is None or n_genes_user > x.shape[1]:
        n_genes_user = x.shape[1]

    # every cell's selected-group index, or k (the remainder: cells in no selected group, NaN included)
    sel = pd.Index(groups_order).get_indexer(col.array)
    codes = np.where(sel >= 0, sel, k).astype(np.int32)
    group_counts = np.bincount(codes, minlength=k + 1)
    n_cells = x.shape[0]

    # --- _basic_stats (:319-452): the t-tests need variances, the Wilcoxon test only means (and pts)
    s, m2, nnz = _ops.rank_genes_group_stats(x, codes, k + 1, expm1_scale=0.0 if mean_in_log_space else log_scale)
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = np.where(group_counts[:, None] > 0, s / group_counts[:, None], 0.0)
        var = m2 / (group_counts[:, None] - 1)
    m2 = np.where(group_counts[:, None] <= 1, 0.0, m2)
    means, variances = mean[:k], var[:k]
    n_sel = group_counts[:k]
    means_rest = vars_rest = pts_rest = None
    if ireference is None:
        n_rest = (n_cells - n_sel)[:, None]
        total = (group_counts[:, None] * mean).sum(axis=0)
        means_rest = (total - n_sel[:, None] * mean[:k]) / n_rest
        if method != "wilcoxon":
            vars_rest = _vars_rest(group_counts.astype(np.float64), mean, m2, k)
        pts_rest = (nnz.sum(axis=0) - nnz[:k]) / n_rest if pts else None
    pts_arr = nnz[:k] / n_sel[:, None] if pts else None

    if method == "wilcoxon":
        results = _wilcoxon(x, codes, k, group_counts, ireference, tie_correct)
    else:
        results = _t_test(method, means, variances, means_rest, vars_rest, n_sel, n_cells, ireference)

    # --- _build_stats_dataframe (:678-740)
    cols: dict = {}
    n_genes_total = x.shape[1]
    for group_index, scores, pvals in results:
        group_name = str(groups_order[group_index])
        scores_sort = np.abs(scores) if rankby_abs else scores
        global_indices = _select_top_n(scores_sort, n_genes_user)
        cols[group_name, "names"] = var_names[global_indices]
        cols[group_name, "scores"] = scores[global_indices]
        cols[group_name, "pvals"] = pvals[global_indices]
        if corr_method == "benjamini-hochberg":
            pvals_adj = _fdr_bh(np.where(np.isnan(pvals), 1.0, pvals))
        else:
            pvals_adj = np.minimum(pvals * n_genes_total, 1.0)
        cols[group_name, "pvals_adj"] = pvals_adj[global_indices]
        mean_group = means[group_index]
        mean_rest = means_rest[group_index] if ireference is None else means[ireference]
        foldchanges = ((expm1_func(mean_group) + 1e-9) / (expm1_func(mean_rest) + 1e-9) if mean_in_log_space
                       else (mean_group + 1e-9) / (mean_rest + 1e-9))
        cols[group_name, "logfoldchanges"] = np.log2(foldchanges[global_indices])
    stats = pd.DataFrame(cols)
    stats.columns = pd.MultiIndex.from_tuples(stats.columns)

    groups_names = [str(name) for name in groups_order]
    if pts_arr is not None:
        adata.uns[key_added]["pts"] = pd.DataFrame(pts_arr.T, index=var_names, columns=groups_names)
    if pts_rest is not None:
        adata.uns[key_added]["pts_rest"] = pd.DataFrame(pts_rest.T, index=var_names, columns=groups_names)
    stats.columns = stats.columns.swaplevel()
    dtypes = {"names": "O", "scores": "float32", "logfoldchanges": "float32", "pvals": "float64", "pvals_adj": "float64"}
    for c in stats.columns.levels[0]:
        adata.uns[key_added][c] = stats[c].to_records(index=False, column_dtypes=dtypes[c])
    log_done(start, f"added to `.uns[{key_added!r}]`")
    return adata if copy else None


def _t_test(method, means, variances, means_rest, vars_rest, n_sel, n_cells, ireference):
    """_RankGenes.t_test (:454-503)."""
    from scipy import stats

    for group_index in range(means.shape[0]):
        if ireference is not None and group_index == ireference:
            continue
        ns_group = int(n_sel[group_index])
        if ireference is not None:
            mean_rest, var_rest, ns_other = means[ireference], variances[ireference], int(n_sel[ireference])
        else:
            mean_rest, var_rest, ns_other = means_rest[group_index], vars_rest[group_index], n_cells - ns_group
        ns_rest = ns_other if method == "t-test" else ns_group
        with np.errstate(invalid="ignore"):
            scores, pvals = stats.ttest_ind_from_stats(mean1=means[group_index], std1=np.sqrt(variances[group_index]),
                                                       nobs1=ns_group, mean2=mean_rest, std2=np.sqrt(var_rest),
                                                       nobs2=ns_rest, equal_var=False)
        scores[np.isnan(scores)] = 0
        pvals[np.isnan(pvals)] = 1
        yield group_index, scores, pvals


def _wilcoxon(x, codes, k, group_counts, ireference, tie_correct):
    """_RankGenes.wilcoxon (:505-579) from the device's exact rank sums and tie terms."""
    from scipy import stats

    rank2, tie = _ops.rank_genes_wilcoxon(x, codes, k + 1, ref=-1 if ireference is None else ireference)
    rank_sums = rank2 / 2.0
    ties = _ops.tie_terms_to_f64(tie)
    n_cells = x.shape[0]
    for group_index in range(k):
        if ireference is not None and group_index == ireference:
            continue
        n_active = int(group_counts[group_index])
        if ireference is None:
            m_active, size, offset = n_cells - n_active, n_cells, n_active * (n_cells + 1) / 2.0
        else:
            m_active = int(group_counts[ireference])
            size, offset = n_active + m_active, n_active * ((n_active + m_active + 1) / 2.0)
            if n_active <= 25 or m_active <= 25:
                logger.info("Few observations in a group for normal approximation (<=25). Lower test accuracy.")
        coef = 1.0
        if tie_correct:
            coef = 1.0 - ties[group_index] / (float(size) ** 3 - size) if size >= 2 else np.ones(x.shape[1])
        with np.errstate(invalid="ignore", divide="ignore"):
            std_dev = np.sqrt(coef * n_active * m_active * (size + 1) / 12.0)
            scores = (rank_sums[group_index] - offset) / std_dev
        scores[np.isnan(scores)] = 0
        pvals = 2 * stats.distributions.norm.sf(np.abs(scores))
        yield group_index, scores, pvals
