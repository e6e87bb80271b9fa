"""Regenerate the rank_genes_groups fixtures from the read-only reference checkout (run in the build container only).

* reference_rank_genes_groups.npz: names and scores of the reference's tests/_data/objs-{t-test,wilcoxon}.npz, pinned by
  its tests/test_rank_genes_groups.py:99-130.
* pbmc68k_reduced_obs.npz: obs/n_counts, obs/bulk_labels (codes, categories) and var/index of the in-tree fixture
  src/scanpy/datasets/10x_pbmc68k_reduced.zarr.zip, to rebuild its `.raw` from the vendored layers/counts and group it.

The zarr arrays are decoded with make_goldens.py's reader; the string arrays (vlen-utf8) with the decoder below.
"""
from __future__ import annotations

import json
import struct
import sys
import zipfile
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent))
from make_goldens import OUT, REF, _zstd_decompress, read_zarr_array  # noqa: E402


def read_zarr_strings(z: zipfile.ZipFile, path: str) -> np.ndarray:
    """A 1-D zarr v3 `string` array (sharded, vlen-utf8 + zstd): each inner chunk is a u32 item count, then a u32
    byte length and the UTF-8 bytes of every item."""
    meta = json.loads(z.read(f"{path}/zarr.json"))
    (n,) = meta["shape"]
    (shard,) = meta["chunk_grid"]["configuration"]["chunk_shape"]
    (inner,) = meta["codecs"][0]["configuration"]["chunk_shape"]
    out: list[str] = [""] * n
    for s in range(-(-n // shard)):
        raw = z.read(f"{path}/c/{s}")
        n_in = shard // inner
        index = raw[-(16 * n_in + 4):-4]
        for k in range(n_in):
            off, nb = struct.unpack_from("<QQ", index, 16 * k)
            if off == 2**64 - 1:
                continue
            buf = _zstd_decompress(raw[off:off + nb])
            (count,) = struct.unpack_from("<I", buf, 0)
            pos, base = 4, s * shard + k * inner
            for i in range(count):
                (ln,) = struct.unpack_from("<I", buf, pos)
                if base + i < n:
                    out[base + i] = buf[pos + 4:pos + 4 + ln].decode("utf-8")
                pos += 4 + ln
    return np.array(out)


def main() -> None:
    gold = {}
    for method in ("t-test", "wilcoxon"):
        with np.load(REF / f"tests/_data/objs-{method}.npz") as f:
            gold[f"{method}_names"] = f["names"].astype(str)
            gold[f"{method}_scores"] = f["scores"]
    np.savez(OUT / "reference_rank_genes_groups.npz", **gold)
    z = zipfile.ZipFile(REF / "src/scanpy/datasets/10x_pbmc68k_reduced.zarr.zip")
    np.savez_compressed(
        OUT / "pbmc68k_reduced_obs.npz", n_counts=read_zarr_array(z, "obs/n_counts"),
        bulk_labels_codes=read_zarr_array(z, "obs/bulk_labels/codes"),
        bulk_labels_categories=read_zarr_strings(z, "obs/bulk_labels/categories"),
        var_index=read_zarr_strings(z, "var/index"))


if __name__ == "__main__":
    main()
