"""tl.rank_genes_groups without a device: the CPU oracle against the reference's goldens and scipy's Mann-Whitney U,
and every argument rule the public function applies before it touches the device."""
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
from scipy import sparse, stats

import scanpy_b200 as sb
from oracle import rank_genes as org
from scanpy_b200._compat import MiniAnnData

GOLDEN = Path(__file__).resolve().parent / "golden"


def pbmc68k_raw():
    """pbmc68k_reduced's `.raw` rebuilt from its vendored `layers/counts` by the reference's recipe
    (src/scanpy/datasets/_datasets.py:409-426) -> (log counts CSR float32 [700 x 765], bulk_labels Categorical, var names)."""
    from scanpy_b200._io import ZarrCSR

    counts = ZarrCSR(GOLDEN / "pbmc68k_reduced_counts.zarr.zip", "layers/counts").tocsr()
    obs = np.load(GOLDEN / "pbmc68k_reduced_obs.npz")
    x = counts.astype(np.float32)
    x.data /= np.repeat(obs["n_counts"] / 1e4, np.diff(x.indptr))
    x.data = np.round(np.log1p(x.data), 3)
    x = x.tolil()
    x[357, 715] = 4.019
    labels = pd.Categorical.from_codes(obs["bulk_labels_codes"].astype(int), categories=list(obs["bulk_labels_categories"]))
    return x.tocsr().astype(np.float32), labels, pd.Index(obs["var_index"])


@pytest.mark.parametrize("method", ["t-test", "wilcoxon"])
def test_oracle_reproduces_reference_goldens(method):
    # the reference's tests/test_rank_genes_groups.py:99-130 (n = 7 for wilcoxon there)
    gold = np.load(GOLDEN / "reference_rank_genes_groups.npz")
    x, labels = org.example_data()
    res = org.rank_genes_groups(x, labels, [0, 1], method=method, n_genes=20)
    n = 7 if method == "wilcoxon" else None
    for g in range(2):
        np.testing.assert_allclose(gold[f"{method}_scores"][g, :n], res[g]["scores"][:n], rtol=1e-5, atol=1e-10)
        np.testing.assert_array_equal(gold[f"{method}_names"][g, :n], res[g]["order"][:n].astype(str))


@pytest.mark.parametrize("reference", ["Dendritic", None])
def test_oracle_tie_corrected_pvals_match_mannwhitneyu(reference):
    x, labels, _ = pbmc68k_raw()
    dense = x.toarray().astype(np.float64)
    lab = np.asarray(labels)
    grp = "CD14+ Monocyte"
    res = org.rank_genes_groups(dense, lab, [grp, "Dendritic"] if reference else [grp], reference=reference,
                                method="wilcoxon", tie_correct=True)[grp]
    pvals = np.empty(dense.shape[1])
    pvals[res["order"]] = res["pvals"]
    a = dense[lab == grp]
    b = dense[lab == reference] if reference else dense[lab != grp]
    checked = 0
    for j in range(dense.shape[1]):
        if np.unique(np.r_[a[:, j], b[:, j]]).size < 2:
            continue  # a constant gene: U's variance is 0 (the oracle, like the reference, reports p = 1)
        p = stats.mannwhitneyu(a[:, j], b[:, j], use_continuity=False, alternative="two-sided", method="asymptotic").pvalue
        np.testing.assert_allclose(pvals[j], p, rtol=1e-5, atol=1e-300)
        checked += 1
    assert checked > 600


def _adata(n=40, g=6, with_raw=False):
    rng = np.random.default_rng(0)
    x = sparse.random(n, g, density=0.5, format="csr", dtype=np.float32, random_state=1)
    ad = MiniAnnData(x)
    ad.obs["grp"] = pd.Categorical(np.repeat(["a", "b", "c", "d"], n // 4))
    ad.obs["str_grp"] = rng.choice(["u", "v"], n)
    if with_raw:
        ad.raw = MiniAnnData(x.copy())
    return ad


def test_argument_errors_match_reference_without_device():
    """tools/_rank_genes_groups.py:881-959 and :240-287: all raised before any device call."""
    tl = sb.tl
    ad = _adata()
    with pytest.raises(ValueError, match=r"Received `use_raw=True`, but `adata.raw` is empty."):
        tl.rank_genes_groups(ad, "grp", use_raw=True)
    with pytest.raises(ValueError, match=r"Method must be one of"):
        tl.rank_genes_groups(ad, "grp", method="t_test")
    with pytest.raises(ValueError, match=r"Correction method must be one of"):
        tl.rank_genes_groups(ad, "grp", corr_method="holm")
    with pytest.raises(ValueError, match="Specify a sequence of groups"):
        tl.rank_genes_groups(ad, "grp", groups="a")
    with pytest.raises(ValueError, match=r"reference = z needs to be one of groupby = \['a', 'b', 'c', 'd'\]."):
        tl.rank_genes_groups(ad, "grp", reference="z")
    with pytest.raises(ValueError, match=r"The shape of the mask do not match the data."):
        tl.rank_genes_groups(ad, "grp", mask_var=np.ones(3, bool))
    for m in ("logreg", "wilcoxon_illico"):
        with pytest.raises(NotImplementedError, match=m):
            tl.rank_genes_groups(ad, "grp", method=m)
    ad_raw = _adata(with_raw=True)
    ad_raw.layers["L"] = ad_raw.X.copy()
    with pytest.raises(ValueError, match=r"Cannot specify `layer` and have `use_raw=True`."):
        tl.rank_genes_groups(ad_raw, "grp", layer="L")
    single = _adata()
    single.obs["grp"] = pd.Categorical(["a"] + ["b"] * 39)
    with pytest.raises(ValueError, match=r"Could not calculate statistics for groups a since they only contain one sample."):
        tl.rank_genes_groups(single, "grp")
    empty = _adata()
    empty.obs["grp"] = pd.Categorical(["b"] * 40, categories=["a", "b"])
    with pytest.raises(ValueError, match=r"Could not calculate statistics for groups a since"):
        tl.rank_genes_groups(empty, "grp")
    many = MiniAnnData(sparse.random(2050, 3, density=0.5, format="csr", dtype=np.float32, random_state=0))
    many.obs["grp"] = pd.Categorical(np.repeat(np.arange(1025).astype(str), 2))
    with pytest.raises(NotImplementedError, match="at most 1024 groups"):
        tl.rank_genes_groups(many, "grp")
    # a string column is made categorical first (sanitize_anndata), so its errors are the categorical ones
    with pytest.raises(ValueError, match=r"reference = w needs to be one of groupby = \['u', 'v'\]."):
        tl.rank_genes_groups(ad, "str_grp", reference="w")
    assert isinstance(ad.obs["str_grp"].dtype, pd.CategoricalDtype)


def test_mini_anndata_raw_and_var_names():
    ad = _adata(with_raw=True)
    assert list(ad.var_names) == [str(i) for i in range(6)]
    c = ad.copy()
    assert c.raw is not None and c.raw is not ad.raw
    assert (c.raw.X != ad.raw.X).nnz == 0
    assert MiniAnnData(np.zeros((2, 2))).raw is None
