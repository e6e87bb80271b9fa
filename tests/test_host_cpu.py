"""CPU-only tests: C-ABI surface, loud failure without a GPU, host-side mirror of the reference's helpers."""
import re
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
from scipy import sparse

import scanpy_b200 as sb
from oracle import knn as oknn
from scanpy_b200 import _abi, pp, tl
from scanpy_b200._compat import LegacyRng, MiniAnnData, accepts_legacy_random_state, seed_from_rng

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "scanpy_b200.h").read_text()
    declared = set(re.findall(r"\b(sb2_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 18
    assert declared == set(_abi.SIGNATURES), declared ^ set(_abi.SIGNATURES)
    lib = _abi.load()
    for name in declared:
        assert hasattr(lib, name)
    assert lib.sb2_version() >= 100


def test_no_cpu_fallback_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_abi.B200Error):
        _abi.Context()
    x = sparse.random(50, 40, density=0.2, format="csr", dtype=np.float32, random_state=0)
    with pytest.raises(_abi.B200Error):
        pp.pca(x, n_comps=5)
    with pytest.raises(_abi.B200Error):  # zero_center=False is served by the device (TruncatedSVD semantics): no CPU path here
        pp.pca(_adata(), zero_center=False)
    # the raw C entry point also refuses (no device) instead of computing on the host
    import ctypes

    h = ctypes.c_void_p()
    rc = _abi.load().sb2_ctx_create(0, None, 0, ctypes.byref(h))
    assert rc != 0 and b"CUDA" in _abi.load().sb2_last_error()


def test_product_never_imports_oracle():
    for py in (ROOT / "scanpy_b200").glob("*.py"):
        src = py.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), py
    for cu in (ROOT / "scanpy_b200" / "csrc").glob("*.cu*"):
        assert "oracle/" not in cu.read_text().replace("// oracle", ""), cu


def test_indices_distances_roundtrip_matches_reference_helpers():
    # src/scanpy/neighbors/_common.py:35-98 ; tests/test_neighbors_common.py:59-103
    rs = np.random.RandomState(0)
    n, k = 40, 6
    idx = np.stack([np.r_[i, rs.permutation(np.delete(np.arange(n), i))[: k - 1]] for i in range(n)])
    dist = np.sort(rs.rand(n, k), axis=1)
    dist[:, 0] = 0
    m = pp._get_sparse_matrix_from_indices_distances(idx, dist, keep_self=False)
    mo = oknn.sparse_from_indices_distances(idx, dist, keep_self=False)
    assert (m != mo).nnz == 0 and (np.diff(m.indptr) == k - 1).all()
    # sklearn style (self stored) -> trimmed to k; RAPIDS style (no self) -> self prepended
    full = pp._get_sparse_matrix_from_indices_distances(idx, dist, keep_self=True)
    i2, d2 = pp._get_indices_distances_from_sparse_matrix(full, k - 1)
    assert i2.shape == (n, k - 1) and (i2[:, 0] == np.arange(n)).all()
    i3, d3 = pp._get_indices_distances_from_sparse_matrix(m, k)
    np.testing.assert_array_equal(i3, idx)
    np.testing.assert_allclose(d3, dist)
    with pytest.raises(AssertionError, match="first neighbor"):
        pp._get_sparse_matrix_from_indices_distances(idx[:, 1:], dist[:, 1:], keep_self=False)
    # ragged rows -> slow path + RuntimeWarning (src/scanpy/neighbors/_common.py:101-123,126-143)
    rag = m.tolil(); rag[0, idx[0, 1]] = 0; rag = rag.tocsr(); rag.eliminate_zeros()
    with pytest.warns(RuntimeWarning, match="no constant number"):
        i4, d4 = pp._get_indices_distances_from_sparse_matrix(rag, k)
    assert i4.shape == (n, k) and (i4[:, 0] == np.arange(n)).all()


def test_random_state_shim():
    # src/scanpy/_utils/random.py:182-208
    @accepts_legacy_random_state(0)
    def f(*, rng=None):
        return rng

    assert isinstance(f(), LegacyRng) and f().arg == 0
    assert f(random_state=7).arg == 7
    assert not isinstance(f(rng=3), LegacyRng)
    with pytest.raises(TypeError):
        f(rng=1, random_state=1)
    assert seed_from_rng(LegacyRng(5)) == 5
    assert seed_from_rng(np.random.default_rng(1)) == seed_from_rng(np.random.default_rng(1))


def _adata(n=30, g=20):
    rs = np.random.RandomState(0)
    return MiniAnnData(sparse.csr_matrix(rs.poisson(1.0, (n, g)).astype(np.float32)))


def test_pca_argument_errors_match_reference():
    a = _adata()
    with pytest.raises(NotImplementedError, match="layer`/`obsm` and `chunked"):
        pp.pca(a, layer="x", chunked=True)  # _pca/__init__.py:201-204
    with pytest.raises(ValueError, match="incompatible with `obsm`"):
        pp.pca(a, mask_var=np.ones(20, bool), obsm="foo")  # :228-230
    with pytest.raises(ValueError, match=r"Did not find `adata.var\['nope'\]`"):
        pp.pca(a, mask_var="nope")  # get/get.py:637-646 ; tests/test_pca.py:405-423
    with pytest.raises(ValueError, match="The shape of the mask do not match the data."):
        pp.pca(a, mask_var=np.ones(7, bool))
    with pytest.raises(ValueError, match="Mask array must be boolean."):
        pp.pca(a, mask_var=np.ones(20, int))
    with pytest.raises(ValueError, match=r"n_components=100 must be between 1 and min\(n_samples, n_features\)=20"):
        pp.pca(a, n_comps=100)  # tests/test_pca.py:292-296
    with pytest.warns(UserWarning, match="Ignoring svd_solver='randomized'"):
        assert pp._solver_code("randomized", n_vars=100) in (0, 1)  # _pca/__init__.py:451-467
    assert pp._solver_code("covariance_eigh", n_vars=10**6) == 1
    assert pp._solver_code(None, n_vars=2000) == 1 and pp._solver_code("arpack", n_vars=30000) == 0


def test_neighbors_and_leiden_argument_errors_match_reference():
    a = _adata()
    with pytest.raises(ValueError, match="`method` needs to be one of"):
        pp.neighbors(a, method="bogus")  # neighbors/__init__.py:742-744
    with pytest.raises(ValueError, match="only with `knn = True`"):
        pp.neighbors(a, knn=False)  # :748-751
    with pytest.raises(ValueError, match="Unknown transformer: nope"):
        pp.neighbors(a, transformer="nope")  # :782-787
    with pytest.raises(ValueError, match="Did not find X_foo"):
        pp._choose_representation(a, use_rep="X_foo", n_pcs=None)  # tools/_utils.py:48-50
    # tests/test_clustering.py:105-127
    with pytest.raises(ValueError, match="flavor must be either 'igraph' or 'leidenalg', but 'foo' was passed"):
        tl.leiden(a, flavor="foo")
    with pytest.raises(ValueError, match="Cannot use igraph’s leiden implementation with a directed graph."):
        tl.leiden(a, flavor="igraph", directed=True)
    with pytest.raises(ValueError, match="Do not pass in partition_type argument when using igraph."):
        tl.leiden(a, flavor="igraph", partition_type=object)
    with pytest.raises(ValueError, match="You need to run `pp.neighbors` first"):
        tl.leiden(a, flavor="igraph")  # _utils/__init__.py:980-985
    with pytest.raises(ValueError, match="both obsp, neighbors_key"):
        tl._choose_graph(a, "x", "y")


def test_transformer_protocol_surface():
    # src/scanpy/neighbors/_types.py:53-64: fit / transform / fit_transform / get_params / set_params
    t = sb.B200KNNTransformer(n_neighbors=7)
    assert t.get_params()["n_neighbors"] == 7
    assert t.set_params(n_neighbors=9) is t and t.get_params()["n_neighbors"] == 9
    for name in ("fit", "transform", "fit_transform"):
        assert callable(getattr(t, name))
    with pytest.raises(NotImplementedError):
        sb.B200KNNTransformer(metric="cosine")


def test_rename_groups_matches_reference():
    # src/scanpy/tools/_utils_clustering.py:16-30 ; tests/test_clustering.py:177-213
    a = _adata(6, 5)
    a.obs["louvain"] = pd.Categorical(["0", "1", "1", "2", "1", "0"])
    adj = sparse.csr_matrix(np.ones((6, 6), np.float32))
    sub, ridx = tl._restrict_adjacency(a, "louvain", restrict_categories=["1"], adjacency=adj)
    assert sub.shape == (3, 3) and ridx.tolist() == [False, True, True, False, True, False]
    out = tl._rename_groups(a, "louvain", restrict_categories=["1"], restrict_indices=ridx, groups=np.array([0, 1, 0]))
    assert out.tolist() == ["0", "1,0", "1,1", "2", "1,0", "0"]
    with pytest.raises(ValueError, match="not a valid category"):
        tl._restrict_adjacency(a, "louvain", restrict_categories=["9"], adjacency=adj)


def test_struct_layouts_match_the_header(tmp_path):
    """The ctypes mirrors of the info structs (scanpy_b200/_abi.py) must have the size and field offsets a C compiler
    gives include/scanpy_b200.h - the header is the contract a reference-side binding would be written against."""
    import ctypes
    import shutil
    import subprocess

    from scanpy_b200 import _abi

    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    root = Path(__file__).resolve().parents[1]
    structs = {"sb2_device_info": _abi.DeviceInfo, "sb2_pca_info": _abi.PcaInfo, "sb2_knn_info": _abi.KnnInfo,
               "sb2_leiden_info": _abi.LeidenInfo, "sb2_eigs_info": _abi.EigsInfo}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "scanpy_b200.h"', "int main(void) {"]
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} %zu", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf(" %zu", offsetof({cname}, {fname}));')
        lines.append('  printf("\\n");')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(root / "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.strip().splitlines()
    for line, (cname, cls) in zip(out, structs.items()):
        parts = line.split()
        assert parts[0] == cname
        assert int(parts[1]) == ctypes.sizeof(cls), cname
        assert [int(x) for x in parts[2:]] == [getattr(cls, f).offset for f, _ in cls._fields_], cname


# ------------------------------------------------------------------------------------------ on-disk CSR reader (f4)
@pytest.mark.parametrize("mode,as_zip", [("raw", False), ("zstd", False), ("sharded", False), ("sharded", True)])
def test_zarr_csr_reader_row_chunks(tmp_path, mode, as_zip):
    """scanpy_b200._io.ZarrCSR against stores written by tests/zarr_writer.py: every codec chain the AnnData zarr-v3 layout
    uses, directory and zip stores, ragged row chunks that straddle inner chunks and shards, empty rows."""
    from scipy import sparse

    import zarr_writer
    from scanpy_b200._io import ZarrCSR, read_zarr_backed

    rng = np.random.default_rng(3)
    x = sparse.random(1503, 257, density=0.04, format="csr", dtype=np.float32, random_state=rng)
    x.data = np.round(x.data * 9 + 1, 3).astype(np.float32)
    x[100:140] = 0  # a run of empty rows
    x.eliminate_zeros()
    target = tmp_path / ("store.zarr.zip" if as_zip else "store.zarr")
    zarr_writer.write_csr_store(target, x, mode=mode, chunk=2048, inner=256, as_zip=as_zip)
    z = ZarrCSR(target)
    assert z.shape == x.shape and z.nnz == x.nnz
    got = z.tocsr()
    assert (got.indptr == x.indptr).all() and (got.indices == x.indices).all() and (got.data == x.data).all()
    seen = 0
    for r0, r1, ip, ix, dt in z.row_chunks(211):
        sub = x[r0:r1]
        assert ip.dtype == np.int64 and ix.dtype == np.int32 and dt.dtype == np.float32 and ip[0] == 0
        assert (ip == sub.indptr).all() and (ix == sub.indices).all() and (dt == sub.data).all()
        seen += r1 - r0
    assert seen == x.shape[0]
    ad = read_zarr_backed(target)
    assert ad.n_obs == 1503 and ad.n_vars == 257
    with pytest.raises(KeyError):
        ZarrCSR(target, "layers/nope")


def test_zarr_csr_reader_on_the_reference_fixture():
    """The reference's own in-tree zarr-v3 fixture (sharded + zstd, written by anndata), whose `layers/counts` and `obsm`
    entries tests/golden keeps byte for byte: `layers/counts` must decode to the same arrays as the independent decoder of
    tests/golden/make_goldens.py."""
    import sys
    import zipfile

    fixture = Path(__file__).resolve().parent / "golden" / "pbmc68k_reduced_counts.zarr.zip"
    sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
    import make_goldens as mg

    from scanpy_b200._io import ZarrCSR

    z = ZarrCSR(fixture, "layers/counts")
    m = z.tocsr()
    zz = zipfile.ZipFile(fixture)
    assert m.shape == (700, 765)
    assert (mg.read_zarr_array(zz, "layers/counts/data") == m.data).all()
    assert (mg.read_zarr_array(zz, "layers/counts/indices") == m.indices).all()
    assert (mg.read_zarr_array(zz, "layers/counts/indptr") == m.indptr).all()
    with pytest.raises(NotImplementedError, match="csr_matrix"):
        ZarrCSR(fixture, "obsm")


# ------------------------------------------------------------------------------------------ widened tools: host contracts
def test_widened_tools_argument_contracts_without_gpu():
    """Everything the widened entry points decide BEFORE they touch the device (reference error texts / rules):
    tl.umap (_umap.py:150-158,217-219), tl.diffmap (_diffmap.py:94-99), tl.paga (_paga.py:108-124), tl.louvain
    (_louvain.py:129-131,177-179), metrics.modularity (_metrics.py:158-176), pp.scale's mask rules (get/get.py:633-651)."""
    x = sparse.random(40, 12, density=0.3, format="csr", dtype=np.float32, random_state=0)
    ad = MiniAnnData(x)
    with pytest.raises(ValueError, match=r"Did not find .uns\['neighbors'\]. Run `sc.pp.neighbors` first."):
        tl.umap(ad)
    with pytest.raises(ValueError, match="You need to run `pp.neighbors` first"):
        tl.diffmap(ad)
    with pytest.raises(ValueError, match="You need to run `pp.neighbors` first"):
        tl.paga(ad)
    with pytest.raises(ValueError, match="You need to run `pp.neighbors` first"):
        tl.louvain(ad)
    # a neighbours entry is enough to get past the first gate
    g = sparse.random(40, 40, density=0.2, format="csr", dtype=np.float32, random_state=1)
    g = (g + g.T).tocsr()
    ad.obsp["connectivities"], ad.obsp["distances"] = g, g.astype(np.float64)
    ad.uns["neighbors"] = dict(connectivities_key="connectivities", distances_key="distances", params=dict(method="umap"))
    with pytest.raises(ValueError, match="Unknown method"):
        tl.umap(ad, method="tsne")
    with pytest.raises(NotImplementedError, match="paga"):
        tl.umap(ad, init_pos="paga")
    with pytest.raises(ValueError, match="init_pos must have shape"):
        tl.umap(ad, init_pos=np.zeros((40, 3), np.float32))
    with pytest.raises(ValueError, match="greater than 2"):
        tl.diffmap(ad, n_comps=2)
    with pytest.raises(ValueError, match="tl.leiden` or `tl.louvain"):
        tl.paga(ad)
    with pytest.raises(KeyError, match="not found"):
        tl.paga(ad, groups="nope")
    ad.obs["grp"] = pd.Categorical(["a", "b"] * 20)
    with pytest.raises(NotImplementedError, match="v1.0"):
        tl.paga(ad, groups="grp", model="v1.0")
    with pytest.raises(ValueError, match="needs to be one of"):
        tl.paga(ad, groups="grp", model="v9")
    with pytest.raises(ValueError, match='`flavor` needs to be "vtraag" or "igraph" or "taynaud"'):
        tl.louvain(ad, flavor="nope")
    with pytest.raises(ValueError, match="only a valid argument when `flavour` is \"vtraag\""):
        tl.louvain(ad, flavor="igraph", partition_type=object)
    with pytest.raises(TypeError, match="`labels` must be provided as array"):
        sb.metrics.modularity(g, "leiden", is_directed=False)
    with pytest.raises(TypeError, match="`is_directed` must be provided"):
        sb.metrics.modularity(g, np.zeros(40, int))
    with pytest.raises(ValueError, match="undirected"):
        sb.metrics.modularity(ad, is_directed=True)
    ad.uns["leiden"] = dict(modularity=0.25)
    assert sb.metrics.modularity(ad, mode="retrieve") == 0.25
    with pytest.raises(ValueError, match="must be a string"):
        sb.metrics.modularity(ad, np.zeros(40, int), mode="update")
    with pytest.raises(ValueError, match="Cannot use refererence for mask without providing anndata"):
        pp.scale(x, mask_obs="cells")
    with pytest.raises(ValueError, match="Mask array must be boolean"):
        pp.scale(x, mask_obs=np.ones(40, int))
    with pytest.raises(ValueError, match="shape of the mask"):
        pp.scale(x, mask_obs=np.ones(7, bool))
    with pytest.raises(NotImplementedError, match="layer"):
        pp.scale(ad, layer="counts")
    # find_ab_params: umap-learn's published defaults for (spread 1.0, min_dist 0.5) and (1.0, 0.1)
    from scanpy_b200._graph_tools import find_ab_params

    a, b = find_ab_params(1.0, 0.5)
    assert a == pytest.approx(0.5830300, rel=1e-5) and b == pytest.approx(1.3341669, rel=1e-5)
    a, b = find_ab_params(1.0, 0.1)
    assert a == pytest.approx(1.5769, rel=1e-3) and b == pytest.approx(0.8951, rel=1e-3)
