"""tl.rank_genes_groups on the device against the reference's goldens, the CPU oracle (oracle/rank_genes.py), the
reference's own behaviour tests (tests/test_rank_genes_groups.py) and exact rank / tie-term arithmetic."""
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
from scipy import sparse, stats

import scanpy_b200 as sb
from oracle import rank_genes as org
from scanpy_b200 import _ops
from scanpy_b200._compat import MiniAnnData
from test_rank_genes_cpu import pbmc68k_raw

pytestmark = pytest.mark.gpu

GOLDEN = Path(__file__).resolve().parent / "golden"


def _example(array_type):
    x, labels = org.example_data()
    ad = MiniAnnData(array_type(x))
    ad.obs["true_groups"] = pd.Categorical(labels)
    return ad


ARRAY_TYPES = {"dense": np.asarray, "csr": sparse.csr_matrix, "csc": sparse.csc_matrix}


@pytest.mark.parametrize("layer", [False, True])
@pytest.mark.parametrize("array_type", sorted(ARRAY_TYPES))
@pytest.mark.parametrize("method", ["t-test", "wilcoxon"])
def test_reference_goldens(method, array_type, layer):
    # tests/test_rank_genes_groups.py:99-171 (results and results_layers)
    gold = np.load(GOLDEN / "reference_rank_genes_groups.npz")
    ad = _example(ARRAY_TYPES[array_type])
    if layer:
        ad.layers["to_test"] = ad.X.copy()
        ad.X = ad.X * 0 if not sparse.issparse(ad.X) else ad.X.multiply(0).tocsr()
    sb.tl.rank_genes_groups(ad, "true_groups", n_genes=20, method=method, layer="to_test" if layer else None)
    res = ad.uns["rank_genes_groups"]
    n = 7 if method == "wilcoxon" else None
    for g in range(2):
        np.testing.assert_allclose(gold[f"{method}_scores"][g, :n], res["scores"][str(g)][:n], rtol=1e-5, atol=1e-10)
        np.testing.assert_array_equal(gold[f"{method}_names"][g, :n], res["names"][str(g)][:n])
    assert res["params"]["use_raw"] is False
    assert res["scores"].dtype["0"] == np.float32 and res["logfoldchanges"].dtype["0"] == np.float32
    assert res["pvals"].dtype["0"] == np.float64 and res["names"].dtype["0"] == object


def _pbmc():
    x, labels, var_names = pbmc68k_raw()
    ad = MiniAnnData(x.copy(), var=pd.DataFrame(index=var_names))
    ad.obs["bulk_labels"] = labels
    ad.raw = MiniAnnData(x, var=pd.DataFrame(index=var_names))
    return ad, x.toarray().astype(np.float64), np.asarray(labels), var_names


def _compare(ad, dense, labels, var_names, groups, *, key="rank_genes_groups", pts=False, mask=None, **kw):
    res = ad.uns[key]
    ref = kw.get("reference")
    x = dense if mask is None else dense[:, mask]
    names = var_names if mask is None else var_names[mask]
    orc = org.rank_genes_groups(x, labels, groups, **kw)
    tol = 1e-5
    for grp, o in orc.items():
        got_scores = res["scores"][grp].astype(np.float64)
        np.testing.assert_allclose(got_scores, o["scores"], rtol=tol, atol=1e-6)
        np.testing.assert_allclose(res["pvals"][grp], o["pvals"], rtol=1e-6, atol=1e-300)
        np.testing.assert_allclose(res["pvals_adj"][grp], o["pvals_adj"], rtol=1e-6, atol=1e-300)
        # gene by gene: where scores tie (e.g. +-inf t-scores of zero-variance genes) the two orders may differ
        lfc = dict(zip(res["names"][grp], res["logfoldchanges"][grp].astype(np.float64)))
        got_lfc = np.array([lfc[nm] for nm in np.asarray(names[o["order"]])])
        finite = np.isfinite(o["logfoldchanges"])
        np.testing.assert_allclose(got_lfc[finite], o["logfoldchanges"][finite], rtol=1e-5, atol=1e-5)
        # names agree wherever the oracle's neighbouring scores are separated by more than the tolerance
        sc = o["scores"]
        key_sc = np.abs(sc) if kw.get("rankby_abs") else sc
        gap = np.abs(np.diff(key_sc))
        sep = np.ones(len(sc), bool)
        close = gap <= tol * np.maximum(np.abs(key_sc[:-1]), 1e-6)
        sep[:-1] &= ~close
        sep[1:] &= ~close
        np.testing.assert_array_equal(np.asarray(res["names"][grp])[sep], np.asarray(names[o["order"]])[sep])
        if pts:
            np.testing.assert_array_equal(res["pts"][grp].to_numpy(), o["pts"])
            if ref is None:
                np.testing.assert_array_equal(res["pts_rest"][grp].to_numpy(), o["pts_rest"])
    if pts and ref is not None:
        assert "pts_rest" not in res


METHODS = [("t-test", False), ("t-test_overestim_var", False), ("wilcoxon", False), ("wilcoxon", True)]


@pytest.mark.parametrize("subset", [False, True])
@pytest.mark.parametrize("reference", ["rest", "Dendritic"])
@pytest.mark.parametrize(("method", "tie_correct"), METHODS)
def test_matches_oracle_on_pbmc68k_raw(method, tie_correct, reference, subset):
    ad, dense, labels, var_names = _pbmc()
    groups = ["CD14+ Monocyte", "CD19+ B"] if subset else "all"
    sb.tl.rank_genes_groups(ad, "bulk_labels", method=method, tie_correct=tie_correct, reference=reference,
                            groups=groups, pts=True)
    assert ad.uns["rank_genes_groups"]["params"]["use_raw"] is True
    cats = list(ad.obs["bulk_labels"].cat.categories)
    sel = cats if groups == "all" else groups + ([reference] if reference != "rest" else [])
    _compare(ad, dense, labels, var_names, sel, pts=True, method=method, tie_correct=tie_correct,
             reference=None if reference == "rest" else reference)


@pytest.mark.parametrize(("method", "tie_correct"), METHODS)
def test_options_match_oracle(method, tie_correct):
    ad, dense, labels, var_names = _pbmc()
    cats = list(ad.obs["bulk_labels"].cat.categories)
    kw = dict(method=method, tie_correct=tie_correct)
    sb.tl.rank_genes_groups(ad, "bulk_labels", rankby_abs=True, corr_method="bonferroni", n_genes=50, **kw)
    _compare(ad, dense, labels, var_names, cats, rankby_abs=True, corr_method="bonferroni", n_genes=50, **kw)
    mask = np.zeros(dense.shape[1], bool)
    mask[::3] = True
    sb.tl.rank_genes_groups(ad, "bulk_labels", mask_var=mask, mean_in_log_space=False, key_added="masked", **kw)
    _compare(ad, dense, labels, var_names, cats, key="masked", mask=mask, mean_in_log_space=False, **kw)
    ad.uns["log1p"] = {"base": 2.0}
    sb.tl.rank_genes_groups(ad, "bulk_labels", reference="Dendritic", mean_in_log_space=False, key_added="b2", **kw)
    _compare(ad, dense, labels, var_names, cats, key="b2", reference="Dendritic", mean_in_log_space=False, log1p_base=2.0,
             **kw)


def test_wilcoxon_symmetry():
    # tests/test_rank_genes_groups.py:224-256
    ad, *_ = _pbmc()
    out = {}
    for grp, ref in (("CD14+ Monocyte", "Dendritic"), ("Dendritic", "CD14+ Monocyte")):
        sb.tl.rank_genes_groups(ad, groupby="bulk_labels", groups=["CD14+ Monocyte", "Dendritic"], reference=ref,
                                method="wilcoxon", rankby_abs=True)
        r = ad.uns["rank_genes_groups"]
        out[grp] = np.stack([np.asarray(r[k][grp], np.float64) for k in ("scores", "logfoldchanges", "pvals", "pvals_adj")], 1)
    assert np.allclose(np.abs(out["CD14+ Monocyte"]), np.abs(out["Dendritic"]))


@pytest.mark.parametrize(("n_genes_add", "n_genes_out_add"), [(0, 0), (2, 1)])
def test_mask_n_genes(n_genes_add, n_genes_out_add):
    # tests/test_rank_genes_groups.py:332-357
    ad, *_ = _pbmc()
    mask_var = np.zeros(765, bool)
    mask_var[:6] = True
    no_genes = int(mask_var.sum()) - 1
    sb.tl.rank_genes_groups(ad, mask_var=mask_var, groupby="bulk_labels", groups=["CD14+ Monocyte", "Dendritic"],
                            reference="CD14+ Monocyte", n_genes=no_genes + n_genes_add, method="wilcoxon", use_raw=True)
    assert len(ad.uns["rank_genes_groups"]["scores"]) == no_genes + n_genes_out_add


@pytest.mark.parametrize("method", ["wilcoxon", "t-test", "t-test_overestim_var"])
@pytest.mark.parametrize(("mean_in_log_space", "expected_logfc"), [(True, -2.0), (False, -1.0)])
def test_mean_in_log_space(method, mean_in_log_space, expected_logfc):
    # tests/test_rank_genes_groups.py:506-556 (float64 input: ranked after the documented cast to float32)
    group_a = np.zeros((10, 5))
    group_a[5:] = np.log(9)
    ad = MiniAnnData(np.concatenate([group_a, np.full((10, 5), np.log(9))]))
    ad.obs["bulk_labels"] = ["a"] * 10 + ["b"] * 10
    with pytest.warns(UserWarning, match="float64 data is ranked after a cast to float32"):
        sb.tl.rank_genes_groups(ad, groupby="bulk_labels", groups=["a"], reference="b", method=method,
                                mean_in_log_space=mean_in_log_space)
    np.testing.assert_equal(ad.uns["rank_genes_groups"]["logfoldchanges"]["a"], expected_logfc)


def test_int_groups_append_reference_and_copy():
    ad, dense, labels, var_names = _pbmc()
    ad.obs["num"] = pd.Categorical(ad.obs["bulk_labels"].cat.codes.astype(str))
    out = sb.tl.rank_genes_groups(ad, "num", groups=[5, 6], reference="9", method="wilcoxon", copy=True)
    assert "rank_genes_groups" not in ad.uns
    assert list(out.uns["rank_genes_groups"]["names"].dtype.names) == ["5", "6"]
    cats = list(ad.obs["bulk_labels"].cat.categories)
    res = org.rank_genes_groups(dense, labels, [cats[5], cats[6], cats[9]], reference=cats[9], method="wilcoxon")
    np.testing.assert_allclose(out.uns["rank_genes_groups"]["scores"]["5"], res[cats[5]]["scores"], rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------ device internals
def _rank_reference(dense, codes, n_codes, ref):
    """2 x rank sums (float, exact below 2**53) and exact tie terms (Python ints) with scipy.stats.rankdata."""
    g = dense.shape[1]
    r2 = np.zeros((n_codes, g))
    ties = np.zeros((n_codes, g), dtype=object)
    for q in range(n_codes):
        if ref >= 0 and q in (ref, n_codes - 1):
            continue
        cells = codes == q if ref >= 0 else np.ones(len(codes), bool)
        sub = np.vstack([dense[codes == q], dense[codes == ref]]) if ref >= 0 else dense
        n_q = int((codes == q).sum())
        for j in range(g):
            r = stats.rankdata(sub[:, j])
            r2[q, j] = 2 * (r[:n_q].sum() if ref >= 0 else r[cells & (codes == q)].sum())
            _, cnt = np.unique(sub[:, j], return_counts=True)
            ties[q, j] = sum(int(c) ** 3 - int(c) for c in cnt)
    return r2, ties


@pytest.mark.parametrize("ref", [-1, 2])
def test_rank_sums_and_ties_are_exact(ref):
    rng = np.random.default_rng(3)
    dense = np.round(rng.normal(0, 1, (3000, 24)) * (rng.random((3000, 24)) < 0.3), 1).astype(np.float32)
    dense[:, 0] = 0                              # all-zero gene
    dense[:, 1] = np.abs(dense[:, 1]) + 1        # non-zero in every cell
    dense[:, 2] = np.where(dense[:, 2] != 0, 0.5, 0)  # all non-zeros tied
    codes = rng.integers(0, 6, 3000).astype(np.int32)
    x = sparse.csr_matrix(dense)
    x.data[::7] = 0                              # stored zeros rank with the implicit ones
    rank2, tie = _ops.rank_genes_wilcoxon(x, codes, 6, ref=ref)
    want_r2, want_ties = _rank_reference(x.toarray().astype(np.float64), codes, 6, ref)
    qs = [q for q in range(6) if ref < 0 or q not in (ref, 5)]
    np.testing.assert_array_equal(rank2[qs].astype(np.float64), want_r2[qs])
    got = _ops.tie_terms_to_int(tie)
    assert all(got[q, j] == want_ties[q, j] for q in qs for j in range(24))


def test_tie_terms_exact_on_synthetic_200k():
    from scanpy_b200._synth import synth_scipy

    x, labels = synth_scipy(200_000, 2000, n_clusters=32, r=16)
    n = x.shape[0]
    tied = x[:, 2].tocsc()
    tied.data[:] = 3.0
    full = sparse.csr_matrix((1.0 + np.arange(n, dtype=np.float32) % 7)[:, None])
    x = sparse.hstack([sparse.csr_matrix((n, 1), dtype=np.float32), full, tied, x[:, 3:]]).tocsr().astype(np.float32)
    codes = np.asarray(labels, np.int32)
    cols = [0, 1, 2, 3, 500, 1999]
    for mat in (x, sparse.csr_matrix(np.asarray(x[:, :64].todense()) - 0.25 * (np.arange(64) % 3))):
        _, tie = _ops.rank_genes_wilcoxon(mat, codes, 33, ref=-1)
        got = _ops.tie_terms_to_int(tie[0])
        sub = mat[:, [c for c in cols if c < mat.shape[1]]].toarray()
        for jj, j in enumerate([c for c in cols if c < mat.shape[1]]):
            col = sub[:, jj]
            _, cnt = np.unique(col, return_counts=True)
            assert got[j] == sum(int(c) ** 3 - int(c) for c in cnt), j


@pytest.mark.parametrize("method", ["t-test", "wilcoxon"])
def test_repeated_calls_are_bit_identical(method):
    ad, *_ = _pbmc()
    outs = []
    for _ in range(2):
        sb.tl.rank_genes_groups(ad, "bulk_labels", method=method, tie_correct=True, pts=True)
        r = ad.uns["rank_genes_groups"]
        outs.append({k: r[k].copy() for k in ("names", "scores", "logfoldchanges", "pvals", "pvals_adj")})
    for k in outs[0]:
        for grp in outs[0][k].dtype.names:
            np.testing.assert_array_equal(outs[0][k][grp], outs[1][k][grp])
