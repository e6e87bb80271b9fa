"""Regenerate tests/golden/*.npz from the read-only reference checkout (run in the build container only).

Two sources, both owned by the reference (scverse/scanpy @ fabadb94):

1. Hand-written golden literals in the reference's own tests, lifted by `ast` (no import of
   scanpy needed): tests/test_pca.py:34-59 (A_list, A_pca, A_svd) and
   tests/test_neighbors.py:23-139 (4-point X, distances, umap connectivities, ...).
2. The in-tree fixture src/scanpy/datasets/10x_pbmc68k_reduced.zarr.zip (zarr v3, sharded,
   zstd): obsm/X_pca, obsp/distances, obsp/connectivities, obs/louvain, uns/neighbors params.
   Decoded with zipfile + libzstd via ctypes (zarr/anndata are not installed here).  Its
   `layers/counts` group is also kept as a store (pbmc68k_reduced_counts.zarr.zip) for the
   zarr reader's test.

Usage:  python tests/golden/make_goldens.py   (writes next to this file)
"""
from __future__ import annotations

import ast
import ctypes
import json
import struct
import zipfile
from pathlib import Path

import numpy as np

REF = Path("/root/reference")
OUT = Path(__file__).resolve().parent


def literals_from(pyfile: Path, names: set[str]) -> dict[str, np.ndarray]:
    tree = ast.parse(pyfile.read_text())
    out = {}
    for node in tree.body:
        if isinstance(node, ast.Assign) and len(node.targets) == 1 and isinstance(node.targets[0], ast.Name):
            name = node.targets[0].id
            if name in names:
                val = node.value
                # np.array([...]) -> take the first positional arg
                if isinstance(val, ast.Call):
                    val = val.args[0]
                out[name] = np.array(ast.literal_eval(val))
    missing = names - set(out)
    if missing:
        raise RuntimeError(f"literals not found in {pyfile}: {missing}")
    return out


_zstd = None


def _zstd_decompress(buf: bytes) -> bytes:
    global _zstd
    if _zstd is None:
        _zstd = ctypes.CDLL("libzstd.so.1")
        _zstd.ZSTD_getFrameContentSize.restype = ctypes.c_ulonglong
        _zstd.ZSTD_getFrameContentSize.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
        _zstd.ZSTD_decompress.restype = ctypes.c_size_t
        _zstd.ZSTD_decompress.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
    size = _zstd.ZSTD_getFrameContentSize(buf, len(buf))
    dst = ctypes.create_string_buffer(size)
    got = _zstd.ZSTD_decompress(dst, size, buf, len(buf))
    assert got == size, (got, size)
    return dst.raw


def read_zarr_array(z: zipfile.ZipFile, path: str) -> np.ndarray:
    meta = json.loads(z.read(f"{path}/zarr.json"))
    shape = tuple(meta["shape"])
    dtype = np.dtype({"float32": "<f4", "float64": "<f8", "int32": "<i4", "int64": "<i8", "int8": "i1",
                      "uint8": "u1", "bool": "?"}[meta["data_type"]])
    shard_shape = tuple(meta["chunk_grid"]["configuration"]["chunk_shape"])
    codec = meta["codecs"][0]
    assert codec["name"] == "sharding_indexed"
    inner = tuple(codec["configuration"]["chunk_shape"])
    out = np.zeros(shape, dtype)
    nshards = [-(-s // c) for s, c in zip(shape, shard_shape)]
    ninner = [c // i for c, i in zip(shard_shape, inner)]
    for sidx in np.ndindex(*nshards):
        key = f"{path}/c/" + "/".join(map(str, sidx))
        try:
            raw = z.read(key)
        except KeyError:
            continue
        n_in = int(np.prod(ninner))
        index = raw[-(16 * n_in + 4):-4]
        for k, iidx in enumerate(np.ndindex(*ninner)):
            off, nb = struct.unpack_from("<QQ", index, 16 * k)
            if off == 2**64 - 1:
                continue
            chunk = np.frombuffer(_zstd_decompress(raw[off:off + nb]), dtype).reshape(inner)
            lo = [s * c + i * ic for s, c, i, ic in zip(sidx, shard_shape, iidx, inner)]
            sl = tuple(slice(l, min(l + ic, sh)) for l, ic, sh in zip(lo, inner, shape))
            out[sl] = chunk[tuple(slice(0, s.stop - s.start) for s in sl)]
    return out


def write_counts_store(z: zipfile.ZipFile) -> None:
    """pbmc68k_reduced_counts.zarr.zip: the fixture's `layers/` entries and `obsm/zarr.json`, byte for byte (the whole
    fixture is 1.7 MB).  Where the archive holds a key more than once, the last copy is the one readers see and keep."""
    names = sorted({i.filename for i in z.infolist() if i.filename.startswith("layers/") or i.filename == "obsm/zarr.json"})
    with zipfile.ZipFile(OUT / "pbmc68k_reduced_counts.zarr.zip", "w") as out:
        for name in names:
            info = z.getinfo(name)
            copy = zipfile.ZipInfo(name, date_time=info.date_time)
            copy.compress_type = info.compress_type
            out.writestr(copy, z.read(name))


def main() -> None:
    pca_l = literals_from(REF / "tests/test_pca.py", {"A_list", "A_pca", "A_svd"})
    nb_l = literals_from(
        REF / "tests/test_neighbors.py",
        {"X", "n_neighbors", "distances_euclidean", "distances_euclidean_all", "connectivities_umap",
         "connectivities_gauss_knn", "connectivities_jaccard"},
    )
    sc_names = {"X_original", "X_scaled_original", "X_centered_original", "X_scaled_original_clipped", "X_for_mask",
                "X_scaled_for_mask", "X_centered_for_mask", "X_scaled_for_mask_clipped"}
    sc_l = literals_from(REF / "tests/test_scaling.py", sc_names)  # tests/test_scaling.py:13-69
    np.savez(OUT / "reference_scaling_literals.npz", **{k: v.astype(np.float64) for k, v in sc_l.items()})
    np.savez(OUT / "reference_test_literals.npz",
             A_list=pca_l["A_list"].astype(np.float64), A_pca=pca_l["A_pca"], A_svd=pca_l["A_svd"],
             X4=nb_l["X"].astype(np.float64), n_neighbors4=np.int64(nb_l["n_neighbors"]),
             distances_euclidean=nb_l["distances_euclidean"],
             distances_euclidean_all=nb_l["distances_euclidean_all"],
             connectivities_umap=nb_l["connectivities_umap"],
             connectivities_gauss_knn=nb_l["connectivities_gauss_knn"],
             connectivities_jaccard=nb_l["connectivities_jaccard"])

    z = zipfile.ZipFile(REF / "src/scanpy/datasets/10x_pbmc68k_reduced.zarr.zip")
    fx = {
        "X_pca": read_zarr_array(z, "obsm/X_pca"),
        "dist_data": read_zarr_array(z, "obsp/distances/data"),
        "dist_indices": read_zarr_array(z, "obsp/distances/indices"),
        "dist_indptr": read_zarr_array(z, "obsp/distances/indptr"),
        "conn_data": read_zarr_array(z, "obsp/connectivities/data"),
        "conn_indices": read_zarr_array(z, "obsp/connectivities/indices"),
        "conn_indptr": read_zarr_array(z, "obsp/connectivities/indptr"),
        "louvain_codes": read_zarr_array(z, "obs/louvain/codes"),
        "X_umap": read_zarr_array(z, "obsm/X_umap"),   # the reference's own sc.tl.umap output on this graph
        "n_neighbors": read_zarr_array(z, "uns/neighbors/params/n_neighbors"),
    }
    np.savez_compressed(OUT / "pbmc68k_reduced_graph.npz", **fx)
    for k, v in fx.items():
        print(k, v.shape, v.dtype)
    write_counts_store(z)

    # --- preprocessing golden (SURVEY 8f row f2): the reference's tests/test_highly_variable_genes.py:379-421 runs
    # filter_cells -> normalize_total(1e4) -> log1p -> highly_variable_genes(flavor='seurat') on pbmc68k_reduced's
    # `.raw.X` and compares with tests/_scripts/seurat_hvg.csv (produced by Seurat in R).  `.raw.X` is rebuilt here
    # exactly as src/scanpy/datasets/_datasets.py:407-425 does (V1 preset).
    import csv

    from scipy import sparse

    counts = sparse.csr_matrix((read_zarr_array(z, "layers/counts/data"), read_zarr_array(z, "layers/counts/indices"),
                                read_zarr_array(z, "layers/counts/indptr")), shape=(700, 765))
    n_counts = read_zarr_array(z, "obs/n_counts")
    size_factors = n_counts / 1e4
    log_counts = counts.astype(np.float32)
    log_counts.data /= np.repeat(size_factors, np.diff(log_counts.indptr))
    log_counts.data = np.log1p(log_counts.data)
    log_counts.data = np.round(log_counts.data, 3)
    log_counts[357, 715] = 4.019
    log_counts = log_counts.tocsr()
    with open(REF / "tests/_scripts/seurat_hvg.csv") as fh:
        rows = list(csv.DictReader(fh))
    np.savez_compressed(
        OUT / "pbmc68k_raw_seurat_hvg.npz",
        raw_data=log_counts.data.astype(np.float32), raw_indices=log_counts.indices.astype(np.int32),
        raw_indptr=log_counts.indptr.astype(np.int32),
        means=np.array([float(r["means"]) for r in rows]), dispersions=np.array([float(r["dispersions"]) for r in rows]),
        dispersions_norm=np.array([float(r["dispersions_norm"]) for r in rows]),
        highly_variable=np.array([r["highly_variable"] == "TRUE" for r in rows]))
    print("raw X", log_counts.shape, log_counts.nnz, "seurat rows", len(rows))


if __name__ == "__main__":
    main()
