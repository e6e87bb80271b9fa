#!/usr/bin/env python
"""bench.py — cells/s of the pca -> neighbors -> leiden hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU arithmetic (rank 0)
    python bench.py --steps K --warmup W --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy

Workload (config.workload): synthetic 1.3M cells x 2000 HVGs CSR (~5 % dense), n_pcs=50, k=15 — the
configuration BASELINE.json's metric is quoted on; it fits one B200.  One "step" = one full pass of the
hot path over that matrix.  `value` = cells/s with the CSR already resident in HBM (CUDA events on the
launching stream, barrier + synchronize on both sides, max over ranks); `e2e` = the same pass through
the public scanpy-signature API (sb.pp.pca / sb.pp.neighbors / sb.tl.leiden) from HOST arrays, all
host<->device copies inside the timed region.  N > 1: cells are row-sharded over ranks (strong scaling:
the matrix is fixed), see scanpy_b200/distributed.py.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

# the numpy / scipy wheels bundle an OpenBLAS built for at most 64 threads: on a box with more cores it warns and can
# crash in large GEMMs ("Bad memory unallocation") unless its pool is capped BEFORE the library loads
os.environ.setdefault("OPENBLAS_NUM_THREADS", str(min(32, os.cpu_count() or 1)))

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "cells/sec end-to-end pca->neighbors->leiden, 1.3M x 2k HVG CSR"
UNIT = "cells/s"


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--n-cells", type=int, default=1_300_000)
    p.add_argument("--n-genes", type=int, default=2000)
    p.add_argument("--n-pcs", type=int, default=50)
    p.add_argument("--k", type=int, default=15)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-sample", action="store_true", help="(internal) print one cpu_reference_sample dict as JSON and exit")
    p.add_argument("--sample-rows", type=int, default=100_000)
    p.add_argument("--knn-queries", type=int, default=8192)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-parity", action="store_true", help="skip the host-side fp64 parity checks after the timed region")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (see dump_outputs)")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be at least 1 and --warmup at least 0")
    return a


def workload_config(a, n_gpus):
    return dict(workload=f"synthetic {a.n_cells} cells x {a.n_genes} HVGs CSR (~5% dense, 32 planted clusters), "
                         f"n_pcs={a.n_pcs} k={a.k} (BASELINE.json configs[2]{'/[3]' if n_gpus > 1 else ''})",
                n_cells=a.n_cells, n_genes=a.n_genes, n_pcs=a.n_pcs, n_neighbors=a.k, leiden="resolution=1, n_iterations=-1",
                parallelism=f"row-sharded x{n_gpus}" if n_gpus > 1 else "single GPU",
                l2="inputs (1.0 GB CSR, 260 MB X_pca) exceed the 126 MB L2; no explicit flush")


# ------------------------------------------------------------------------------------------------
# reference CPU arithmetic on a bounded sample (the oracle: sklearn ARPACK PCA and brute kNN are the
# reference's own call sites; fuzzy set / Leiden are the restatements in oracle/)
def _all_cores():
    """BLAS / OpenMP threads = every core of the box, whatever the launcher exported (torch.distributed.run forces
    OMP_NUM_THREADS=1 into its workers, which would otherwise cut the CPU arm to a single thread)."""
    n = int(os.environ.get("SB2_CPU_THREADS", min(os.cpu_count() or 1, 32)))
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        from threadpoolctl import threadpool_limits

        # sklearn's brute-force kNN runs one BLAS call per OpenMP thread: the bundled OpenBLAS builds abort when too many
        # threads call into them at once, so OpenMP gets n threads and every caller a single BLAS thread
        threadpool_limits(limits=n, user_api="openmp")
        threadpool_limits(limits=1, user_api="blas")
    except Exception:
        pass
    try:
        import torch

        torch.set_num_threads(n)
    except Exception:
        pass
    return n


def note(msg: str) -> None:
    """progress marker on stderr (the ONE JSON line owns stdout)"""
    sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
    sys.stderr.flush()


def cpu_reference_sample(a, sample_rows: int = 100_000, knn_queries: int = 8192):
    """Times the reference path on a bounded sample of the workload and scales each stage to n_cells with its own
    complexity (SURVEY.md 8d):
      PCA / connectivities / Leiden: rows [0, sample_rows) of the workload, linear in n;
      exact brute-force kNN: `knn_queries` query rows against ALL n_cells candidate points (the sample's embedding tiled
      to n_cells rows - brute force does not care about the values - so cache behaviour and the per-query cost are the
      real ones), linear in the number of queries."""
    import torch

    from oracle import fuzzy as ofz, knn as oknn, leiden as old, pca as opca
    from scanpy_b200._synth import synth_scipy

    cores = _all_cores()
    n, s = a.n_cells, min(sample_rows, a.n_cells)
    dev = "cuda" if torch.cuda.is_available() else "cpu"  # data generation only
    x, _ = synth_scipy(n, a.n_genes, device=dev, row_stop=s)
    t = time.perf_counter(); p = opca.pca_arpack(x, a.n_pcs); t_pca = time.perf_counter() - t
    xp = p["X_pca"]
    reps = -(-n // s)
    rs = np.random.RandomState(0)
    cand = np.tile(xp, (reps, 1))[:n]
    cand += (1e-3 * rs.standard_normal(cand.shape)).astype(cand.dtype)   # no exact duplicates
    q = min(knn_queries, n)
    from sklearn.neighbors import NearestNeighbors
    nn = NearestNeighbors(n_neighbors=a.k, algorithm="brute", metric="euclidean", n_jobs=-1).fit(cand)
    t = time.perf_counter(); nn.kneighbors(cand[:q]); t_q = time.perf_counter() - t
    pair_rate = q * float(n) / t_q                # distance pairs per second on this host at the real candidate count
    idx, dist = oknn.knn_brute(xp, a.k)          # untimed: inputs for the graph stages
    t = time.perf_counter(); c, _, _ = ofz.fuzzy_simplicial_set(idx, dist, s, a.k); t_fz = time.perf_counter() - t
    t = time.perf_counter(); old.leiden(c, seed=0); t_ld = time.perf_counter() - t
    scale = n / s
    est = dict(pca=t_pca * scale, knn=n * float(n) / pair_rate, connectivities=t_fz * scale, leiden=t_ld * scale)
    total = sum(est.values())
    return dict(value=n / total, unit=UNIT, cores=cores, kind="port",
                sample=(f"rows [0,{s}) of the workload: sklearn PCA(arpack) {t_pca:.2f}s, oracle fuzzy set {t_fz:.2f}s, oracle Leiden "
                        f"{t_ld:.2f}s; sklearn brute kNN {q} queries x {n} points {t_q:.2f}s ({pair_rate:.3g} pairs/s); scaled to {n} cells "
                        f"(PCA/graph/Leiden linear in n, kNN linear in the queries): "
                        + ", ".join(f"{k}={v:.1f}s" for k, v in est.items())),
                stage_seconds_extrapolated=est)


def cpu_reference_subprocess(a, sample_rows: int | None = None, knn_queries: int | None = None):
    """cpu_reference_sample in a FRESH interpreter: thread-pool sizes are fixed by the environment before numpy / scipy /
    sklearn / torch load their BLAS and OpenMP runtimes (inside this process torch has already loaded its own, and the
    launcher may have exported OMP_NUM_THREADS=1), and a crash of a CPU library cannot take the bench line with it."""
    cmd = [sys.executable, str(ROOT / "bench.py"), "--cpu-sample", "--n-cells", str(a.n_cells), "--n-genes", str(a.n_genes),
           "--n-pcs", str(a.n_pcs), "--k", str(a.k)]
    if sample_rows:
        cmd += ["--sample-rows", str(sample_rows)]
    if knn_queries:
        cmd += ["--knn-queries", str(knn_queries)]
    err = ""
    # sklearn's brute-force kNN calls BLAS from every OpenMP thread; the OpenBLAS builds bundled with numpy / scipy abort
    # ("too many memory regions") beyond a few dozen concurrent callers, so: OpenMP threads = min(cores, 32), one BLAS
    # thread per caller - and fewer if even that fails on this host
    for omp in (32, 16, 8):
        omp = min(omp, os.cpu_count() or 1)
        env = dict(os.environ, OMP_NUM_THREADS=str(omp), OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1",
                   CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", ""), SB2_CPU_THREADS=str(omp))
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
            env.pop(k, None)
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        err = f"rc {r.returncode}: {r.stderr.strip()[-200:]}"
    return dict(value=None, unit=UNIT, kind="port", error=f"cpu sample failed ({err})")


def run_reference(a, rank, world):
    if rank != 0:
        return
    t0 = time.perf_counter()
    for _ in range(max(a.warmup, 0)):
        cpu_reference_subprocess(a, sample_rows=8000, knn_queries=256)  # warm the page cache cheaply
    vals = [v for v in (cpu_reference_subprocess(a) for _ in range(max(a.steps, 1))) if v.get("value")]
    if not vals:
        emit(json.dumps(dict(impl="reference", unavailable="the CPU sample failed on this host")))
        return
    order = sorted(vals, key=lambda r: r["value"])
    med = order[len(order) // 2]
    v = float(med["value"])
    ms = 1e3 * a.n_cells / v
    emit(json.dumps(dict(impl="reference", metric=METRIC, value=v, unit=UNIT, n_gpus=a.gpus, steps=a.steps,
                          warmup=a.warmup, ms_per_step=ms, higher_is_better=True, scaling="strong", vs_baseline=None,
                          dtype="f32", data="synthetic", config=workload_config(a, a.gpus),
                          cpu_baseline=dict(med, value=v, runs=[r["value"] for r in vals],
                                            note="value = median of the runs; exact-kNN reference pipeline (sklearn ARPACK PCA + sklearn brute "
                                                 "kNN + oracle fuzzy set / Leiden); scanpy's default approximate kNN (pynndescent) is not installable here"),
                          e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                          wall_s=time.perf_counter() - t0)))


# ------------------------------------------------------------------------------------------------
def parity_checks(a, out, x_host, labels, row_range, n_rows_sample: int = 2000):
    """Host-side parity of the step's OUTPUTS at the bench workload itself (after the timed region, rank 0), against
    float64 oracles (the only place besides cpu_baseline where bench.py touches oracle/):
      knn_sampled_mismatch   rows (of n_rows_sample random query rows) whose neighbour SET differs from a float64 brute
                             force over all n points of the same embedding (0 = identical sets)
      pca_rel_err_vs_f64_gram  per-component relative error (up to sign) of X_pca on the sampled rows against the float64
                             covariance-eigh ground truth (single GPU only: needs the whole CSR on this host)
      ari_vs_planted         adjusted Rand index of the Leiden labels against the generator's planted clusters
      labels_sha1            hash of the membership vector: identical across N = 1, 2, 4, 8 runs of the same code"""
    import hashlib

    from sklearn.metrics import adjusted_rand_score

    from oracle import knn as oknn, pca as opca
    from scanpy_b200 import _ops

    t0 = time.perf_counter()
    res = {}
    member = _ops._to_host(out["membership"])
    res["labels_sha1"] = hashlib.sha1(np.ascontiguousarray(member).tobytes()).hexdigest()[:16]
    xp = _ops._to_host(out["X_pca"])                      # all rows (all-gathered when sharded)
    idx = _ops._to_host(out["knn_idx"])
    n = xp.shape[0]
    rows = np.sort(np.random.RandomState(0).choice(n, min(n_rows_sample, n), replace=False))
    oi, od = oknn.knn_exact_f64(xp, rows, a.k, chunk=128)
    bad = oknn.exact_set_mismatches(idx[rows], oi, od, a.k)
    res["knn_sampled_rows"] = int(len(rows))
    res["knn_sampled_mismatch"] = int(bad.sum())
    res["knn_oracle"] = "float64 brute force over all points (oracle.knn.knn_exact_f64), exact-tie aware"
    if labels is not None:   # this rank's rows (all rows on a single GPU)
        res["ari_vs_planted"] = float(adjusted_rand_score(labels, member[row_range[0]:row_range[1]]))
    if x_host is not None:
        truth = opca.pca_gram_f64(x_host, a.n_pcs, rows=rows)
        got = opca.align_signs(xp[rows].astype(np.float64), truth["X_pca"])
        rel = np.linalg.norm(got - truth["X_pca"], axis=0) / np.linalg.norm(truth["X_pca"], axis=0)
        res["pca_rel_err_vs_f64_gram"] = dict(max=float(rel.max()), median=float(np.median(rel)), n_components=int(len(rel)),
                                              rows=int(len(rows)), spectrum_gap_min=float(truth["gaps"].min()),
                                              variance_rel_err_max=float(np.max(np.abs(out["pca"]["variance"] - truth["variance"]) / truth["variance"])))
    res["seconds"] = time.perf_counter() - t0
    return res


DUMP_BYTES = 64 << 20


def dump_outputs(a, out, directory):
    """Writes what one step of the timed path returns to a caller, as DIR/<name>.npy in float32 or float64, so that two
    builds run with the same arguments (hence the same synthetic input) can be compared output for output.  Per-cell
    outputs are kept for a seeded sample of cells that depends on --n-cells alone (`rows`, sorted), sized so that the
    files stay under 64 MiB; the connectivities are those rows of the CSR with their column indices sorted."""
    import torch
    from scipy import sparse

    from scanpy_b200 import _ops

    n, d, k, g = a.n_cells, a.n_pcs, a.k, a.n_genes
    fixed = 4 * d * g + 8 * g + 16 * d + 8
    per_row = 8 + 4 * d + 16 * k + 8 + 12 * 4 * k    # row id, X_pca, kNN indices + distances, label, ~4k connectivities
    m = min(n, max(1, (DUMP_BYTES - fixed) // per_row))
    rows = np.sort(np.random.RandomState(0).choice(n, m, replace=False))
    sel = torch.from_numpy(rows).to("cuda")
    x_pca, knn_idx, knn_dist, member = _ops._to_host(out["X_pca"].index_select(0, sel), out["knn_idx"].index_select(0, sel),
                                                     out["knn_dist"].index_select(0, sel), out["membership"].index_select(0, sel))
    indptr, indices, data = _ops._to_host(*out["conn"])
    conn = sparse.csr_matrix((data, indices, indptr), shape=(n, n))[rows].sorted_indices()
    pca = out["pca"]
    arrays = dict(rows=rows.astype(np.float64), X_pca=x_pca, pca_components=_ops._to_host(pca["components"]),
                  pca_variance=pca["variance"], pca_variance_ratio=pca["variance_ratio"], pca_mean=pca["mean"],
                  knn_indices=knn_idx.astype(np.float64), knn_distances=knn_dist,
                  connectivities_indptr=conn.indptr.astype(np.float64), connectivities_indices=conn.indices.astype(np.float64),
                  connectivities_data=conn.data, leiden_membership=member.astype(np.float64),
                  modularity=np.float64(out["modularity"]))
    total = sum(np.asarray(v).nbytes for v in arrays.values())
    if total > DUMP_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, v in arrays.items():
        v = np.asarray(v)
        assert v.dtype in (np.float32, np.float64), (name, v.dtype)
        np.save(os.path.join(directory, f"{name}.npy"), v)
    note(f"dumped {len(arrays)} outputs ({total / 2**20:.1f} MiB, {m} of {n} cells) to {directory}")


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu, self.rows, self._stop_ev = gpu_index, [], threading.Event()

    def run(self):
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_ev.wait(0.2)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=5)
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for j, nm in enumerate(names) if any(len(r) > 5 + j and r[5 + j].lower().startswith("active") for r in self.rows)]
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=float(self.rows[0][2]) if self.rows[0][2].replace(".", "").isdigit() else None,
                    power_w_max=max((float(r[3]) for r in self.rows if r[3].replace(".", "").isdigit()), default=None),
                    samples=len(self.rows), reasons=reasons)


def run_b200(a, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import scanpy_b200 as sb
    from scanpy_b200 import _abi, _ops, distributed as sbd
    from scanpy_b200._synth import synth_scipy

    torch.cuda.set_device(local_rank)
    ctx = _abi.default_context()
    if world > 1:
        sbd.attach_comm(ctx)
    n, g = a.n_cells, a.n_genes
    bounds = sbd.shard_bounds(n, world)
    r0, r1 = bounds[rank]
    x_local, labels_local = synth_scipy(n, g, device="cuda", row_start=r0, row_stop=r1)   # this rank's CSR rows (host)
    d_csr = _ops.csr_to_device(x_local)
    torch.cuda.synchronize()

    def step():
        return sbd.pipeline_sharded(ctx, *d_csr, bounds, rank, g, n_pcs=a.n_pcs, n_neighbors=a.k, solver=1, seed=0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    note(f"rank {rank}: data resident, warm-up")
    for _ in range(a.warmup):
        out = step()
    barrier()
    note("timed region")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        out = step()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = (ctx.launches - launches0) // max(a.steps, 1)
    clocks = sampler.stop() if sampler else None
    if world > 1:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / a.steps
    value = n / (ms_step / 1e3)

    # ---- e2e through the public API from host arrays: every step copies its inputs host -> device (from page-locked
    # host memory, as the contract prescribes) and its results device -> host inside the timed region ----
    def pinned_csr(x):
        from scipy import sparse

        def pin(arr):
            t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
            return t.numpy()   # a view: the array keeps the pinned tensor alive
        return sparse.csr_matrix((pin(x.data), pin(x.indices), pin(x.indptr)), shape=x.shape, copy=False)

    note(f"timed region done: {ms_step:.1f} ms/step; e2e")
    e2e = None
    if not a.no_e2e:
        reps = max(1, a.steps)
        x_pinned = pinned_csr(x_local)
        if world == 1:
            ad = sb.MiniAnnData(x_pinned)  # the input object exists before the timed region (like a loaded .h5ad)

            def e2e_step():
                sb.pp.pca(ad, n_comps=a.n_pcs)
                sb.pp.neighbors(ad, n_neighbors=a.k)
                sb.tl.leiden(ad, flavor="igraph", n_iterations=-1)
                return ad
            e2e_step()  # warm-up (pinned staging buffers, pools)
            torch.cuda.synchronize()
            _ops.TRANSFER.update(h2d=0, d2h=0)
            t0 = time.perf_counter()
            for _ in range(reps):
                ad = e2e_step()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / reps
            e2e = dict(value=n / dt, unit=UNIT, h2d_bytes_per_step=_ops.TRANSFER["h2d"] // reps,
                       d2h_bytes_per_step=_ops.TRANSFER["d2h"] // reps, s_per_step=dt, reps=reps,
                       api="sb.pp.pca -> sb.pp.neighbors -> sb.tl.leiden on a host MiniAnnData (scipy CSR in page-locked host memory in, "
                           "numpy/scipy/pandas out; X_pca and the connectivities stay resident on the device between the three calls)")
        else:
            # sharded e2e: host CSR shard -> device, pipeline, membership + X_pca shard back to host
            def e2e_step():
                d = _ops.csr_to_device(x_pinned)
                o = sbd.pipeline_sharded(ctx, *d, bounds, rank, g, n_pcs=a.n_pcs, n_neighbors=a.k, solver=1, seed=0)
                return _ops._to_host(o["membership"]), _ops._to_host(o["X_pca_local"])
            e2e_step()
            barrier()
            _ops.TRANSFER.update(h2d=0, d2h=0)
            t0 = time.perf_counter()
            for _ in range(reps):
                e2e_step()
            barrier()
            dt = torch.tensor([(time.perf_counter() - t0) / reps], device="cuda", dtype=torch.float64)
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            e2e = dict(value=n / float(dt.item()), unit=UNIT, h2d_bytes_per_step=_ops.TRANSFER["h2d"] // reps,
                       d2h_bytes_per_step=_ops.TRANSFER["d2h"] // reps, s_per_step=float(dt.item()), reps=reps,
                       api="scanpy_b200.distributed.pipeline_sharded from per-rank host CSR shards in page-locked memory (bytes are per rank)")

    if rank != 0:
        return
    if a.dump_outputs:
        dump_outputs(a, out, a.dump_outputs)
    peaks = {}
    try:
        peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
    except Exception:
        pass
    ki = out["knn_info"]
    ach = ki["pass1_flops"] / (ki["pass1_ms"] * 1e-3) / 1e12
    issued = ki["pass1_issued_flops"] / (ki["pass1_ms"] * 1e-3) / 1e12
    peak_tensor = peaks.get("bf16_tflops_sustained", 1400.0)
    sm_max = (clocks or {}).get("sm_max_mhz") or 1965.0
    if ki["pass1_tensor"]:
        # DRAM bytes per launch of the dominant kernel from the committed ncu capture of this exact workload
        # (profiles/r1_ncu_metrics_knn_tiered.txt: dram__bytes_read 12.388 GB + dram__bytes_write 0.780 GB)
        traffic = 11.973e9 if (world == 1 and a.n_cells == 1_300_000 and a.n_pcs == 50 and a.k == 15) else None
        roofline = dict(bound="tensor", kernel="knn_pass1_tc_kernel", achieved=ach, peak=peak_tensor, unit="TFLOP/s",
                        frac=ach / peak_tensor, traffic=traffic,
                        traffic_source=("profiles/r2_ncu_metrics_knn_sweep2_meanfront.txt (ncu --set full of knn_sweep2_kernel, main launch, dram read + write; algorithmic operand bytes: "
                                        "0.33 GB of fp16 images)" if traffic else None),
                        peak_source=("MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained"),
                        launch_ms=ki["pass1_ms"], algorithmic_flops_per_launch=ki["pass1_flops"],
                        issued_tensor_tflops=issued, frac_issued=issued / peak_tensor,
                        note=("achieved counts the ALGORITHMIC 2*n_q*n*d flops of the pairwise-distance sweep over the summed duration "
                              "of its launches (pilot wave + rest; rows the fp16 tier cannot certify are swept again in split "
                              "precision, n_resweep of them). The fp16 tier issues K = d+3 padded to 64 instead of 50, plus a 1/16 "
                              "sample of the candidate tiles for the starting threshold: issued_tensor_tflops / frac_issued say how "
                              "busy the tensor pipe is. Each 256x128 score tile is 8 MMAs (512 tensor cycles) against one TMEM "
                              "hand-off + 4 tcgen05.ld round trips per epilogue warp, so the sweep is paced by the accumulator "
                              "hand-off, not by the MMAs (DESIGN.md section 5)"),
                        n_resweep=ki.get("n_resweep", 0),
                        share_of_step=ki["pass1_ms"] / ms_step)
    else:
        fp32_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12
        roofline = dict(bound="tensor", kernel="knn_pass1_kernel", achieved=ach, peak=peak_tensor, unit="TFLOP/s",
                        frac=ach / peak_tensor, traffic=None, launch_ms=ki["pass1_ms"], algorithmic_flops_per_launch=ki["pass1_flops"],
                        note=f"fp32 FFMA path (d too large for the tensor-core tiles); CUDA-core ceiling {fp32_peak:.1f} TFLOP/s",
                        frac_fp32_ffma=ach / fp32_peak, share_of_step=ki["pass1_ms"] / ms_step)
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup, ms_per_step=ms_step,
                higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32", data="synthetic",
                config=workload_config(a, world), e2e=e2e, gpu_launches=int(launches), clocks=clocks, roofline=roofline,
                stages=dict(pca_iterations=out["pca"]["iterations"], pca_converged=out["pca"]["converged"],
                            knn_uncertified_rows=ki["n_uncertified"], knn_resweep_rows=ki.get("n_resweep", 0), leiden=out["leiden_info"], n_communities=out["n_communities"],
                            modularity=out["modularity"]))
    # per-stage device times of ONE extra, untimed step (CUDA events between the stages of pipeline_sharded on rank 0): where
    # the step goes at this N - the replicated stages (connectivities, leiden, the dense part of pca) are the serial fraction
    try:
        evs = []
        sbd.pipeline_sharded(ctx, *d_csr, bounds, rank, g, n_pcs=a.n_pcs, n_neighbors=a.k, solver=1, seed=0, stage_events=evs)
        barrier()
        line["stages"]["stage_ms"] = {name: round(evs[i - 1][1].elapsed_time(ev), 3) for i, (name, ev) in enumerate(evs) if i > 0}
    except Exception as exc:  # never lose the bench line over a diagnostic
        line["stages"]["stage_ms"] = {"error": repr(exc)[:200]}
    note("parity checks")
    if not a.no_parity:
        line["stages"]["parity"] = parity_checks(a, out, x_local if world == 1 else None, labels_local, (r0, r1))
    if world == 1 and not a.no_cpu_baseline:
        note("cpu baseline sample")
        line["cpu_baseline"] = cpu_reference_subprocess(a)
    emit(json.dumps(line))


_REAL_STDOUT = None


def emit(line: str) -> None:
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, library chatter) was diverted."""
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (line + "\n").encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # native libraries that print to fd 1 (e.g. "NCCL version ...") now land on stderr
    a = parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if a.cpu_sample:
        emit(json.dumps(cpu_reference_sample(a, sample_rows=a.sample_rows, knn_queries=a.knn_queries)))
        return
    if a.impl == "reference":
        os.environ["OMP_NUM_THREADS"] = str(min(64, os.cpu_count() or 1))   # before sklearn / torch load their OpenMP runtimes
        os.environ.pop("MKL_NUM_THREADS", None)
        os.environ.pop("OPENBLAS_NUM_THREADS", None)
        run_reference(a, rank, world)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl")
    try:
        run_b200(a, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
