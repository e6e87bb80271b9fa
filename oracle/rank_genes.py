"""CPU oracle of sc.tl.rank_genes_groups (t-test, t-test_overestim_var, wilcoxon).
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): never imported by scanpy_b200/.

An independent numpy/scipy restatement of src/scanpy/tools/_rank_genes_groups.py that shares none of the device
path's shortcuts: group and rest statistics are computed directly from the dense cells of each side, ranks come from
`scipy.stats.rankdata` and tie corrections from `scipy.stats.tiecorrect`, per gene column.  The Benjamini-Hochberg
correction (statsmodels' `fdr_bh`, not installed here) and the top-n selection (:42-49) are restated.
"""
from __future__ import annotations

import numpy as np
from scipy import stats


def fdr_bh(pvals: np.ndarray) -> np.ndarray:
    order = np.argsort(pvals)
    n = len(pvals)
    adj = pvals[order] * n / np.arange(1, n + 1)
    adj = np.minimum.accumulate(adj[::-1])[::-1]
    out = np.empty(n)
    out[order] = np.minimum(adj, 1.0)
    return out


def select_top_n(scores: np.ndarray, n_top: int) -> np.ndarray:
    partition = np.argpartition(scores, -n_top)[-n_top:]
    return np.arange(scores.shape[0])[partition][np.argsort(scores[partition])[::-1]]


def wilcoxon_columns(x_group: np.ndarray, x_other: np.ndarray):
    """Rank sums of the group's cells and tie terms sum(t^3 - t) of every column of vstack(group, other)."""
    both = np.vstack([x_group, x_other])
    n_g = x_group.shape[0]
    rank_sums = np.empty(both.shape[1])
    ties = np.empty(both.shape[1])
    tc = np.empty(both.shape[1])
    for j in range(both.shape[1]):
        r = stats.rankdata(both[:, j])
        rank_sums[j] = r[:n_g].sum()
        _, cnt = np.unique(both[:, j], return_counts=True)
        ties[j] = float((cnt.astype(np.float64) ** 3 - cnt).sum())
        tc[j] = stats.tiecorrect(r)
    return rank_sums, ties, tc


def rank_genes_groups(x: np.ndarray, labels: np.ndarray, groups: list, *, reference=None, method: str = "t-test",
                      tie_correct: bool = False, corr_method: str = "benjamini-hochberg", n_genes: int | None = None,
                      rankby_abs: bool = False, mean_in_log_space: bool = True, log1p_base=None) -> dict:
    """x dense [n, g] (float64 of the values the device reads), labels [n] group label per cell.
    -> {group: dict(order, scores, pvals, pvals_adj, logfoldchanges, pts, pts_rest)}, each indexed by `order` (the
    top-n gene indices) except pts / pts_rest (all genes)."""
    x = np.asarray(x, dtype=np.float64)
    expm1 = (lambda v: np.expm1(v * np.log(log1p_base))) if log1p_base is not None else np.expm1
    xs = x if mean_in_log_space else expm1(x)
    n_top = x.shape[1] if n_genes is None or n_genes > x.shape[1] else n_genes
    out = {}
    for grp in groups:
        if reference is not None and grp == reference:
            continue
        in_g = labels == grp
        rest = (labels == reference) if reference is not None else ~in_g
        a, b = xs[in_g], xs[rest]
        n_a, n_b = a.shape[0], b.shape[0]
        if method in ("t-test", "t-test_overestim_var"):
            with np.errstate(invalid="ignore", divide="ignore"):
                scores, pvals = stats.ttest_ind_from_stats(
                    a.mean(0), np.sqrt(a.var(0, ddof=1)), n_a, b.mean(0), np.sqrt(b.var(0, ddof=1)),
                    n_b if method == "t-test" else n_a, equal_var=False)
            scores[np.isnan(scores)] = 0
            pvals[np.isnan(pvals)] = 1
        else:
            rank_sums, _, tc = wilcoxon_columns(x[in_g], x[rest])
            coef = tc if tie_correct else 1.0
            with np.errstate(invalid="ignore", divide="ignore"):
                scores = (rank_sums - n_a * (n_a + n_b + 1) / 2.0) / np.sqrt(coef * n_a * n_b * (n_a + n_b + 1) / 12.0)
            scores[np.isnan(scores)] = 0
            pvals = 2 * stats.norm.sf(np.abs(scores))
        order = select_top_n(np.abs(scores) if rankby_abs else scores, n_top)
        adj = fdr_bh(np.where(np.isnan(pvals), 1.0, pvals)) if corr_method == "benjamini-hochberg" else \
            np.minimum(pvals * x.shape[1], 1.0)
        m_a, m_b = a.mean(0), b.mean(0)
        fc = (expm1(m_a) + 1e-9) / (expm1(m_b) + 1e-9) if mean_in_log_space else (m_a + 1e-9) / (m_b + 1e-9)
        out[grp] = dict(order=order, scores=scores[order], pvals=pvals[order], pvals_adj=adj[order],
                        logfoldchanges=np.log2(fc[order]), pts=(x[in_g] != 0).mean(0),
                        pts_rest=(x[~in_g] != 0).mean(0))
    return out


def example_data(seed: int = 1234) -> tuple[np.ndarray, np.ndarray]:
    """The reference's tests/test_rank_genes_groups.py:40-61 example (rng = RandomState(seed), as its _LegacyRng wraps):
    100 x 20 counts, group 0 = the first 10 cells with planted markers in genes 0..4."""
    rng = np.random.RandomState(seed)
    x = rng.binomial(1, 0.15, (100, 20)) * rng.negative_binomial(2, 0.25, (100, 20))
    x[0:10, 0:5] = rng.binomial(1, 0.9, (10, 5)) * rng.negative_binomial(1, 0.5, (10, 5))
    labels = np.concatenate((np.zeros(10, dtype=int), np.ones(90, dtype=int)))
    return x, labels
