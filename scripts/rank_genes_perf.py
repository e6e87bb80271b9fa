"""tl.rank_genes_groups at config C (1.3M cells x 2000 genes, 32 planted clusters as `groupby`) on one GPU.

Prints, for t-test, Wilcoxon vs rest (tie_correct=True) and Wilcoxon vs the largest group:
* per-stage device times (CUDA events; grouped statistics, radix sort, rank walk) on CSR arrays already resident in HBM,
  median of 5 after one warm-up call, and achieved bytes/s against the algorithmic byte model below;
* the wall time of the public call (median of 3 after a warm-up), which INCLUDES uploading the host CSR;
* a check of 32 sampled genes (4 groups) against the CPU oracle at full size;
* the CPU oracle's Wilcoxon ranking time on a 20-gene slab, scaled to 2000 genes (an extrapolation, not a measurement).
Byte model (from shapes): grouped statistics = 2 passes x 8 B per stored entry (column index + value); sort = passes x
24 B per stored entry (8 B key read twice - histogram and scatter - and written once); rank walk ~ 8 B per entry.
Usage: python scripts/rank_genes_perf.py [out.txt]
"""
import subprocess
import sys
import time
from ctypes import c_float
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import torch  # noqa: E402
from scipy import stats  # noqa: E402

import scanpy_b200 as sb  # noqa: E402
from oracle import rank_genes as org  # noqa: E402
from scanpy_b200 import _abi, _ops  # noqa: E402
from scanpy_b200._abi import check, ptr  # noqa: E402
from scanpy_b200._synth import synth_scipy  # noqa: E402

lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def main():
    out = Path(sys.argv[1]) if len(sys.argv) > 1 else None
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU path")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout.strip()
    say(f"card: {card}")
    n, g, k = 1_300_000, 2000, 32
    x, labels = synth_scipy(n, g, n_clusters=k)
    nnz = int(x.nnz)
    say(f"config C: {n} cells x {g} genes, nnz {nnz}, {k} planted clusters")
    ctx = _abi.default_context()
    d_indptr, d_indices, d_data = _ops.csr_to_device(x)
    codes_all = np.asarray(labels, np.int32)
    sizes = np.bincount(codes_all, minlength=k)
    largest = int(np.argmax(sizes))

    def ev_time(fn, reps=5):
        ts = []
        fn()
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    # grouped statistics on resident arrays
    codes = np.where(codes_all >= 0, codes_all, k).astype(np.int32)
    rows = _ops._to_device(np.argsort(codes, kind="stable").astype(np.int32))
    offsets = np.zeros(k + 2, np.int64)
    np.cumsum(np.bincount(codes, minlength=k + 1), out=offsets[1:])
    s = torch.empty((k + 1, g), dtype=torch.float64, device="cuda")
    m2, cnt = torch.empty_like(s), torch.empty((k + 1, g), dtype=torch.int64, device="cuda")
    stats_ms = ev_time(lambda: check(ctx.lib.sb2_rank_genes_group_stats(
        ctx.handle, n, g, ptr(d_indptr), ptr(d_indices), ptr(d_data), ptr(rows), ptr(offsets), k + 1, 0.0, ptr(s),
        ptr(m2), ptr(cnt))))
    stats_bytes = 2 * 8 * nnz
    say(f"grouped statistics (t-test; 2 passes): {stats_ms:.2f} ms device, {stats_bytes / stats_ms / 1e6:.0f} GB/s "
        f"against {stats_bytes / 1e9:.2f} GB modelled")

    d_codes = _ops._to_device(codes)
    d_sizes = _ops._to_device(np.bincount(codes, minlength=k + 1).astype(np.int64))
    rank2 = torch.empty((k + 1, g), dtype=torch.int64, device="cuda")
    tie = torch.empty((k + 1, g, 2), dtype=torch.int64, device="cuda")
    for label, ref in (("wilcoxon vs rest", -1), (f"wilcoxon vs largest group ({largest}, {sizes[largest]} cells)", largest)):
        ms = (c_float * 2)()
        per = []
        for rep in range(6):
            check(ctx.lib.sb2_rank_genes_wilcoxon(ctx.handle, n, g, ptr(d_indptr), ptr(d_indices), ptr(d_data), nnz,
                                                  ptr(d_codes), ptr(d_sizes), k + 1, ref, ptr(rank2), ptr(tie), ms))
            if rep:
                per.append((ms[0], ms[1]))
        sort_ms, walk_ms = np.median([p[0] for p in per]), np.median([p[1] for p in per])
        say(f"{label}: sort {sort_ms:.2f} ms (incl. key build), rank walk {walk_ms:.2f} ms (device, median of 5)")
        for passes in (6, 7):
            b = passes * 24 * nnz
            say(f"  sort at {passes} passes x 24 B/entry = {b / 1e9:.1f} GB -> {b / sort_ms / 1e6:.0f} GB/s achieved")

    ad = sb.MiniAnnData(x)
    ad.obs["clusters"] = pd.Categorical.from_codes(codes_all, categories=[str(i) for i in range(k)])
    walls = {}
    for name, kw in (("t-test", dict(method="t-test")), ("wilcoxon rest tie_correct", dict(method="wilcoxon", tie_correct=True)),
                     ("wilcoxon vs largest", dict(method="wilcoxon", reference=str(largest)))):
        sb.tl.rank_genes_groups(ad, "clusters", key_added=name, **kw)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            sb.tl.rank_genes_groups(ad, "clusters", key_added=name, **kw)
            ts.append(time.perf_counter() - t0)
        walls[name] = float(np.median(ts))
        say(f"public call {name}: {walls[name] * 1e3:.0f} ms wall (median of 3; includes the host CSR upload)")

    # 32 sampled genes, 4 groups, at full size against the CPU oracle
    rng = np.random.default_rng(0)
    genes = np.sort(rng.choice(g, 32, replace=False))
    dense = x[:, genes].toarray().astype(np.float64)
    groups = [str(i) for i in range(4)]
    lab = np.asarray(ad.obs["clusters"]).astype(str)
    worst = 0.0
    for name, kw in (("t-test", dict(method="t-test")), ("wilcoxon rest tie_correct", dict(method="wilcoxon", tie_correct=True))):
        orc = org.rank_genes_groups(dense, lab, groups, **kw)
        r = ad.uns[name]
        for grp in groups:
            pos = {int(v): i for i, v in enumerate(r["names"][grp])}
            got = np.array([r["scores"][grp][pos[int(j)]] for j in genes], np.float64)
            want = np.empty(32)
            want[orc[grp]["order"]] = orc[grp]["scores"]
            worst = max(worst, float(np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-6))))
    say(f"oracle check, 32 sampled genes x 4 groups at full size (t-test, wilcoxon+tie_correct): max rel. score error {worst:.2e}")

    slab = x[:, :20].toarray()
    t0 = time.perf_counter()
    stats.rankdata(slab, axis=0)
    cpu = time.perf_counter() - t0
    say(f"CPU oracle ranking (scipy rankdata, 1 core) of a 20-gene slab: {cpu:.2f} s -> {cpu * 100:.0f} s for 2000 genes "
        "(EXTRAPOLATED x100, not measured)")
    if out is not None:
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
