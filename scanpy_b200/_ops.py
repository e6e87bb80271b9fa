"""Host-side drivers of the C-ABI kernels: numpy/scipy in, numpy/scipy out.

Each function stages its inputs in (pinned) host memory, copies them to the device with torch,
calls ONE C-ABI entry point of libscanpy_b200.so (include/scanpy_b200.h) and copies the results
back.  torch is plumbing only (allocation, copies, stream); there is no CPU code path.
`*_device` variants take/return torch CUDA tensors so a pipeline can keep intermediates in HBM.
"""
from __future__ import annotations

from ctypes import byref, c_double, c_int32, c_int64

import numpy as np

from . import _abi
from ._abi import EigsInfo, KnnInfo, LeidenInfo, PcaInfo, check, ptr


def _torch():
    import torch

    return torch


TRANSFER = dict(h2d=0, d2h=0)  # bytes moved by the host-array entry points (bench.py's e2e accounting)


def _to_host(*tensors):
    """CUDA tensors -> numpy arrays through PINNED destination buffers (a pageable `.cpu()` runs at ~3.5 GB/s,
    a pinned async copy at PCIe speed); all copies are enqueued first, then one synchronize."""
    torch = _torch()
    outs = []
    for t in tensors:
        TRANSFER["d2h"] += t.numel() * t.element_size()
        if t.numel() == 0:
            outs.append(torch.empty(t.shape, dtype=t.dtype))
            continue
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t, non_blocking=True)
        outs.append(h)
    torch.cuda.current_stream().synchronize()
    arrs = [h.numpy() for h in outs]
    return arrs[0] if len(arrs) == 1 else arrs


def _to_device(arr: np.ndarray, *, pin: bool = True):
    """numpy -> CUDA tensor (async H2D on the current stream).  Arrays that already live in page-locked memory (the caller
    pinned or registered them) are copied straight from where they are; pageable arrays go through a pinned staging
    buffer (torch's caching host allocator keeps it across calls)."""
    torch = _torch()
    t = torch.from_numpy(np.ascontiguousarray(arr))
    TRANSFER["h2d"] += t.numel() * t.element_size()
    if pin and t.numel() > 0 and not t.is_pinned():
        try:
            t = t.pin_memory()
        except RuntimeError:
            pass
    return t.to("cuda", non_blocking=True)


class _Resident:
    """Device twins of the most recent host-side results, so that the next stage of the path (pca -> neighbors -> leiden
    through the scanpy-signature API) does not upload what the previous stage just downloaded.  Keyed by the identity
    of the host buffer (address, size, dtype) plus a sampled checksum, so a buffer the user has rewritten in place is
    uploaded again instead of being trusted.  SB2_RESIDENT=0 disables it.  Holds at most 4 entries."""

    def __init__(self):
        self._items: dict = {}

    @staticmethod
    def _key(a: np.ndarray):
        return (a.__array_interface__["data"][0], a.nbytes, a.dtype.str)

    @staticmethod
    def _probe(a: np.ndarray) -> int:
        flat = a.reshape(-1).view(np.uint8)
        step = max(1, flat.size // 4096)
        return hash(flat[::step][:8192].tobytes())

    def put(self, host: np.ndarray, dev) -> None:
        import os

        if os.environ.get("SB2_RESIDENT", "1") == "0" or not isinstance(host, np.ndarray) or not host.flags.c_contiguous:
            return
        if len(self._items) >= 4:
            self._items.pop(next(iter(self._items)))
        self._items[self._key(host)] = (self._probe(host), dev)

    def get(self, host):
        if not isinstance(host, np.ndarray) or not host.flags.c_contiguous:
            return None
        hit = self._items.get(self._key(host))
        if hit is None or hit[0] != self._probe(host):
            return None
        return hit[1]

    def clear(self) -> None:
        self._items.clear()


RESIDENT = _Resident()


def csr_to_device(x):
    """scipy CSR (float32/float64 data, any index width) -> (indptr int64, indices int32, data float32) CUDA tensors."""
    hit = RESIDENT.get(x.data) if x.data.dtype == np.float32 else None
    if hit is not None and len(hit) == 3 and hit[0].numel() == x.shape[0] + 1 and hit[2].numel() == x.nnz:
        return hit
    indptr = np.asarray(x.indptr, dtype=np.int64)
    indices = np.asarray(x.indices, dtype=np.int32)
    data = np.asarray(x.data, dtype=np.float32)
    return _to_device(indptr), _to_device(indices), _to_device(data)


# ------------------------------------------------------------------------------------------ PCA
def pca_csr_device(ctx, d_indptr, d_indices, d_data, n: int, g: int, n_comps: int, *, solver: int = 0,
                   max_iter: int = 0, tol: float = 0.0, seed: int = 0, n_total: int | None = None):
    torch = _torch()
    x_pca = torch.empty((n, n_comps), dtype=torch.float32, device="cuda")
    comps = torch.empty((n_comps, g), dtype=torch.float32, device="cuda")
    var = np.empty(n_comps, np.float64)
    ratio = np.empty(n_comps, np.float64)
    mean = np.empty(g, np.float64)
    info = PcaInfo()
    check(ctx.lib.sb2_pca_csr_f32(ctx.handle, n, n if n_total is None else n_total, g, ptr(d_indptr), ptr(d_indices),
                                  ptr(d_data), n_comps, solver, max_iter, tol, seed, ptr(x_pca), ptr(comps),
                                  ptr(var), ptr(ratio), ptr(mean), byref(info)))
    return dict(X_pca=x_pca, components=comps, variance=var, variance_ratio=ratio, mean=mean,
                iterations=info.iterations, converged=bool(info.converged), max_rel_residual=info.max_rel_residual,
                total_var=info.total_var)


OVERLAP_MIN_NNZ = 1 << 24   # below ~16.7M stored entries the upload is too short to be worth pipelining


def _pca_csr_overlapped(ctx, x, n_comps: int, seed: int, n_chunks: int = 8):
    """Gram-route PCA of a HOST scipy CSR with the upload hidden behind the first pass over the data: the CSR arrays go up
    in `n_chunks` row ranges on a side stream, and as each range lands the compute stream adds its column statistics and
    Gram matrix (sb2_pca_stream_accumulate_f32 - the out-of-core entry point, pointed at the resident arrays).  The
    projection then runs over the whole resident matrix.  Same arithmetic as solver 1 up to the fp64 summation order.
    OPT-IN (SB2_PCA_OVERLAP=1): measured on B200 at 1.3M x 2000 from page-locked arrays, pca() takes 78 ms of wall time
    this way against 62 ms of device work, but the bench's e2e did not improve (0.489 s vs 0.471 s without it, within
    box-to-box noise) - the 21 ms upload is already a small part of the step - so the plain upload stays the default."""
    torch = _torch()
    n, g = x.shape
    nnz = int(x.nnz)
    main = torch.cuda.current_stream()
    side = _side_stream()
    indptr64 = np.asarray(x.indptr, dtype=np.int64)
    h_idx = torch.from_numpy(np.ascontiguousarray(x.indices, dtype=np.int32))
    h_dat = torch.from_numpy(np.ascontiguousarray(x.data, dtype=np.float32))
    d_indptr = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    d_indices = torch.empty(nnz, dtype=torch.int32, device="cuda")
    d_data = torch.empty(nnz, dtype=torch.float32, device="cuda")
    stats = torch.zeros(2 * g, dtype=torch.float64, device="cuda")
    gram = torch.zeros((g, g), dtype=torch.float64, device="cuda")
    cuts = np.unique(np.r_[0, np.searchsorted(indptr64, np.linspace(0, nnz, n_chunks + 1)[1:-1]), n]).astype(np.int64)
    side.wait_stream(main)   # the fresh allocations above may recycle blocks still in use on the compute stream
    pending = []
    with torch.cuda.stream(side):
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            lo, hi = int(indptr64[r0]), int(indptr64[r1])
            ip = torch.from_numpy(indptr64[r0:r1 + 1] - lo)
            parts = []
            for dst, src in ((d_indices[lo:hi], h_idx[lo:hi]), (d_data[lo:hi], h_dat[lo:hi])):
                if src.numel() and not src.is_pinned():
                    src = src.pin_memory()
                dst.copy_(src, non_blocking=True)
                parts.append(src)
            ipp = ip.pin_memory()
            d_ip = ipp.to("cuda", non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(side)
            pending.append((int(r0), int(r1), lo, hi, d_ip, ev, (parts, ipp)))
        hp = torch.from_numpy(indptr64)
        hp = hp if hp.is_pinned() else hp.pin_memory()
        d_indptr.copy_(hp, non_blocking=True)
        ev_all = torch.cuda.Event()
        ev_all.record(side)
    TRANSFER["h2d"] += nnz * 8 + (n + 1) * 8 + (n + len(pending)) * 8
    for r0, r1, lo, hi, d_ip, ev, _keep in pending:
        main.wait_event(ev)
        d_ip.record_stream(main)
        check(ctx.lib.sb2_pca_stream_accumulate_f32(ctx.handle, r1 - r0, g, ptr(d_ip), ptr(d_indices[lo:hi]) if hi > lo else ptr(d_indices),
                                                    ptr(d_data[lo:hi]) if hi > lo else ptr(d_data), ptr(stats), ptr(gram)))
    comps = torch.empty((n_comps, g), dtype=torch.float32, device="cuda")
    proj = torch.empty(g * 128, dtype=torch.float32, device="cuda")
    shift = torch.empty(128, dtype=torch.float32, device="cuda")
    var = np.empty(n_comps, np.float64)
    ratio = np.empty(n_comps, np.float64)
    mean = np.empty(g, np.float64)
    l = c_int32()
    info = PcaInfo()
    check(ctx.lib.sb2_pca_stream_solve_f32(ctx.handle, n, g, ptr(stats), ptr(gram), n_comps, 0, 0.0, seed, ptr(comps), ptr(var),
                                           ptr(ratio), ptr(mean), ptr(proj), ptr(shift), byref(l), byref(info)))
    main.wait_event(ev_all)
    x_pca = torch.empty((n, n_comps), dtype=torch.float32, device="cuda")
    check(ctx.lib.sb2_pca_stream_project_f32(ctx.handle, n, g, ptr(d_indptr), ptr(d_indices), ptr(d_data), n_comps, l.value, ptr(proj),
                                             ptr(shift), ptr(x_pca)))
    for t in (d_indptr, d_indices, d_data):
        t.record_stream(side)
    return dict(X_pca=x_pca, components=comps, variance=var, variance_ratio=ratio, mean=mean, iterations=info.iterations,
                converged=bool(info.converged), max_rel_residual=info.max_rel_residual, total_var=info.total_var)


_SIDE = {}


def _side_stream():
    torch = _torch()
    dev = torch.cuda.current_device()
    if dev not in _SIDE:
        _SIDE[dev] = torch.cuda.Stream(device=dev)
    return _SIDE[dev]


def pca_csr(x, n_comps: int, *, solver: int = 0, max_iter: int = 0, tol: float = 0.0, seed: int = 0, ctx=None):
    """Top-n_comps PCA of a scipy CSR matrix; host arrays out (X_pca float32 [n,k], components float32 [k,g])."""
    import os

    ctx = ctx or _abi.default_context()
    n, g = x.shape
    min_nnz = int(os.environ.get("SB2_PCA_OVERLAP_MIN_NNZ", OVERLAP_MIN_NNZ))
    if (solver == 1 and max_iter == 0 and tol == 0.0 and x.nnz >= min_nnz and getattr(ctx, "n_ranks", 1) == 1
            and g >= 64 and os.environ.get("SB2_PCA_OVERLAP", "0") == "1"):
        out = _pca_csr_overlapped(ctx, x, n_comps, seed)
        d_x_pca = out["X_pca"]
        out["X_pca"], out["components"] = _to_host(out["X_pca"], out["components"])
        RESIDENT.put(out["X_pca"], d_x_pca)
        return out
    d_indptr, d_indices, d_data = csr_to_device(x)
    out = pca_csr_device(ctx, d_indptr, d_indices, d_data, n, g, n_comps, solver=solver, max_iter=max_iter, tol=tol,
                         seed=seed)
    d_x_pca = out["X_pca"]
    out["X_pca"], out["components"] = _to_host(out["X_pca"], out["components"])
    RESIDENT.put(out["X_pca"], d_x_pca)
    return out


def tsvd_csr(x, n_comps: int, *, solver: int = 1, seed: int = 0, ctx=None):
    """Truncated SVD of a scipy CSR (no centring; `sc.pp.pca(zero_center=False)`): host arrays out, keys as `pca_csr`."""
    torch = _torch()
    ctx = ctx or _abi.default_context()
    n, g = x.shape
    d_indptr, d_indices, d_data = csr_to_device(x)
    x_pca = torch.empty((n, n_comps), dtype=torch.float32, device="cuda")
    comps = torch.empty((n_comps, g), dtype=torch.float32, device="cuda")
    var = np.empty(n_comps, np.float64)
    ratio = np.empty(n_comps, np.float64)
    info = PcaInfo()
    check(ctx.lib.sb2_tsvd_csr_f32(ctx.handle, n, g, ptr(d_indptr), ptr(d_indices), ptr(d_data), n_comps, solver, 0, 0.0, seed,
                                   ptr(x_pca), ptr(comps), ptr(var), ptr(ratio), byref(info)))
    h_x, h_c = _to_host(x_pca, comps)
    RESIDENT.put(h_x, x_pca)
    return dict(X_pca=h_x, components=h_c, variance=var, variance_ratio=ratio, iterations=info.iterations,
                converged=bool(info.converged), max_rel_residual=info.max_rel_residual, total_var=info.total_var)


def pca_csr_chunked(x, n_comps: int, *, chunk_size: int, seed: int = 0, ctx=None):
    """Out-of-core PCA of a host scipy CSR: the rows stream through the device `chunk_size` at a time (two passes: Gram
    accumulation, projection); device memory holds one chunk + the g x g Gram matrix.  Same outputs as `pca_csr`."""
    torch = _torch()
    ctx = ctx or _abi.default_context()
    n, g = x.shape
    chunk_size = max(1, int(chunk_size))
    stats = torch.zeros(2 * g, dtype=torch.float64, device="cuda")
    gram = torch.zeros((g, g), dtype=torch.float64, device="cuda")

    def chunks():
        if hasattr(x, "row_chunks"):   # on-disk matrix (scanpy_b200._io.ZarrCSR): only the chunk is ever in host memory
            for r0, r1, indptr, indices, data in x.row_chunks(chunk_size):
                yield r0, r1, _to_device(indptr), _to_device(indices), _to_device(data)
            return
        for r0 in range(0, n, chunk_size):
            r1 = min(n, r0 + chunk_size)
            lo, hi = int(x.indptr[r0]), int(x.indptr[r1])
            indptr = np.asarray(x.indptr[r0:r1 + 1], dtype=np.int64) - lo
            yield r0, r1, _to_device(indptr), _to_device(np.asarray(x.indices[lo:hi], dtype=np.int32)), \
                _to_device(np.asarray(x.data[lo:hi], dtype=np.float32))

    for r0, r1, dp, di, dd in chunks():
        check(ctx.lib.sb2_pca_stream_accumulate_f32(ctx.handle, r1 - r0, g, ptr(dp), ptr(di), ptr(dd), ptr(stats), ptr(gram)))
    comps = torch.empty((n_comps, g), dtype=torch.float32, device="cuda")
    proj = torch.empty(g * 128, dtype=torch.float32, device="cuda")
    shift = torch.empty(128, dtype=torch.float32, device="cuda")
    var = np.empty(n_comps, np.float64)
    ratio = np.empty(n_comps, np.float64)
    mean = np.empty(g, np.float64)
    l = c_int32()
    info = PcaInfo()
    check(ctx.lib.sb2_pca_stream_solve_f32(ctx.handle, n, g, ptr(stats), ptr(gram), n_comps, 0, 0.0, seed, ptr(comps), ptr(var),
                                           ptr(ratio), ptr(mean), ptr(proj), ptr(shift), byref(l), byref(info)))
    x_pca = np.empty((n, n_comps), np.float32)
    for r0, r1, dp, di, dd in chunks():
        part = torch.empty((r1 - r0, n_comps), dtype=torch.float32, device="cuda")
        check(ctx.lib.sb2_pca_stream_project_f32(ctx.handle, r1 - r0, g, ptr(dp), ptr(di), ptr(dd), n_comps, l.value, ptr(proj),
                                                 ptr(shift), ptr(part)))
        x_pca[r0:r1] = _to_host(part)
    return dict(X_pca=x_pca, components=_to_host(comps), variance=var, variance_ratio=ratio, mean=mean,
                iterations=info.iterations, converged=bool(info.converged), max_rel_residual=info.max_rel_residual,
                total_var=info.total_var)


# ------------------------------------------------------------------------------------------ kNN
def knn_device(ctx, d_x, n_neighbors: int, *, q0: int = 0, n_query: int | None = None):
    torch = _torch()
    if d_x.dtype != torch.float32 or not d_x.is_contiguous() or d_x.dim() != 2:
        raise TypeError("knn_device expects a contiguous 2-D float32 CUDA tensor")
    n, d = d_x.shape
    n_query = n - q0 if n_query is None else n_query
    idx = torch.empty((n_query, n_neighbors), dtype=torch.int32, device="cuda")
    dist = torch.empty((n_query, n_neighbors), dtype=torch.float64, device="cuda")
    info = KnnInfo()
    check(ctx.lib.sb2_knn_l2_f32(ctx.handle, n, d, ptr(d_x), q0, n_query, n_neighbors, ptr(idx), ptr(dist),
                                 byref(info)))
    return idx, dist, dict(n_uncertified=int(info.n_uncertified), max_norm=float(info.max_norm),
                           pass1_ms=float(info.pass1_ms), pass1_flops=float(info.pass1_flops),
                           pass1_issued_flops=float(info.pass1_issued_flops), pass1_tensor=int(info.pass1_tensor), n_resweep=int(info.n_resweep))


def knn(x: np.ndarray, n_neighbors: int, *, ctx=None):
    """Exact euclidean kNN incl. self in column 0 -> (indices int32 [n,k], distances float64 [n,k], info)."""
    ctx = ctx or _abi.default_context()
    d_x = _to_device(np.asarray(x, dtype=np.float32))
    idx, dist, info = knn_device(ctx, d_x, n_neighbors)
    h_idx, h_dist = _to_host(idx, dist)
    return h_idx, h_dist, info


# ------------------------------------------------------------------------------------------ graph
def fuzzy_simplicial_set_device(ctx, d_idx, d_dist, n: int, k: int, *, set_op_mix_ratio: float = 1.0,
                                local_connectivity: float = 1.0):
    torch = _torch()
    cap = 2 * n * max(k - 1, 1)
    indptr = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    indices = torch.empty(cap, dtype=torch.int32, device="cuda")
    data = torch.empty(cap, dtype=torch.float32, device="cuda")
    sig = torch.empty(n, dtype=torch.float32, device="cuda")
    rho = torch.empty(n, dtype=torch.float32, device="cuda")
    nnz = c_int64()
    check(ctx.lib.sb2_fuzzy_simplicial_set_f32(ctx.handle, n, k, ptr(d_idx), ptr(d_dist), set_op_mix_ratio,
                                               local_connectivity, ptr(indptr), ptr(indices), ptr(data), cap,
                                               byref(nnz), ptr(sig), ptr(rho)))
    m = nnz.value
    return indptr, indices[:m], data[:m], sig, rho


def fuzzy_simplicial_set(knn_indices: np.ndarray, knn_dists: np.ndarray, *, ctx=None, **kw):
    """-> scipy CSR float32 connectivities (symmetric, sorted indices, no explicit zeros)."""
    from scipy import sparse

    ctx = ctx or _abi.default_context()
    n, k = knn_indices.shape
    d_idx = _to_device(np.asarray(knn_indices, dtype=np.int32))
    d_dist = _to_device(np.asarray(knn_dists, dtype=np.float64))
    indptr, indices, data, sig, rho = fuzzy_simplicial_set_device(ctx, d_idx, d_dist, n, k, **kw)
    ip, h_data, h_indices, h_sig, h_rho = _to_host(indptr, data, indices, sig, rho)
    c = sparse.csr_matrix((h_data, h_indices, ip if ip[-1] >= 2**31 else ip.astype(np.int32)), shape=(n, n))
    return c, h_sig, h_rho


def knn_connectivities(knn_indices: np.ndarray, knn_dists: np.ndarray, method: str, *, ctx=None):
    """method='gauss' | 'jaccard' connectivities from k-lists -> scipy CSR float64 (sorted, no explicit zeros)."""
    from scipy import sparse

    torch = _torch()
    ctx = ctx or _abi.default_context()
    n, k = knn_indices.shape
    d_idx = _to_device(np.asarray(knn_indices, dtype=np.int32))
    d_dist = _to_device(np.asarray(knn_dists, dtype=np.float64))
    cap = 2 * n * max(k - 1, 1)
    indptr = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    indices = torch.empty(cap, dtype=torch.int32, device="cuda")
    data = torch.empty(cap, dtype=torch.float64, device="cuda")
    nnz = c_int64()
    check(ctx.lib.sb2_knn_connectivities_f64(ctx.handle, n, k, ptr(d_idx), ptr(d_dist), {"gauss": 1, "jaccard": 2}[method],
                                             ptr(indptr), ptr(indices), ptr(data), cap, byref(nnz)))
    m = nnz.value
    ip, h_data, h_indices = _to_host(indptr, data[:m].contiguous(), indices[:m].contiguous())
    return sparse.csr_matrix((h_data, h_indices, ip if ip[-1] >= 2**31 else ip.astype(np.int32)), shape=(n, n))


def knn_and_connectivities(x: np.ndarray, n_neighbors: int, *, ctx=None):
    """Exact kNN + UMAP connectivities with the (idx, dist) lists kept on the device in between.
    -> (distances scipy CSR float64 [n,n] with k-1 entries per row: the self column is dropped ON THE DEVICE, so the
    host never re-strides the n x k lists; connectivities scipy CSR float32)."""
    from scipy import sparse

    ctx = ctx or _abi.default_context()
    x = np.ascontiguousarray(x, dtype=np.float32)  # the kernel reads float32 rows: never reinterpret another dtype
    n = x.shape[0]
    d_x = RESIDENT.get(x)
    if d_x is None or tuple(d_x.shape) != tuple(x.shape):
        d_x = _to_device(x)
    d_idx, d_dist, _ = knn_device(ctx, d_x, n_neighbors)
    indptr, indices, data, _, _ = fuzzy_simplicial_set_device(ctx, d_idx, d_dist, n, n_neighbors)
    # column 0 is the query itself by construction (knn_rescore_kernel / knn_fallback_kernel), cf. the reference's
    # `_get_sparse_matrix_from_indices_distances(..., keep_self=False)` (src/scanpy/neighbors/_common.py:35-61)
    nb_idx = d_idx[:, 1:].contiguous().view(-1)
    nb_dist = d_dist[:, 1:].contiguous().view(-1)
    ip, h_data, h_indices, h_nb_idx, h_nb_dist = _to_host(indptr, data, indices, nb_idx, nb_dist)
    conn = sparse.csr_matrix((h_data, h_indices, ip if ip[-1] >= 2**31 else ip.astype(np.int32)), shape=(n, n))
    RESIDENT.put(conn.data, (indptr, indices, data))
    km1 = n_neighbors - 1
    it = np.int64 if n * km1 >= 2**31 else np.int32
    dist_indptr = np.arange(0, n * km1 + 1, km1, dtype=it) if km1 > 0 else np.zeros(n + 1, it)
    dist = sparse.csr_matrix((h_nb_dist, h_nb_idx, dist_indptr), shape=(n, n))
    return dist, conn


def leiden_device(ctx, d_indptr, d_indices, d_weights, n: int, *, resolution: float = 1.0, n_iterations: int = -1,
                  seed: int = 0):
    torch = _torch()
    member = torch.empty(n, dtype=torch.int32, device="cuda")
    q = c_double()
    nc = c_int32()
    info = LeidenInfo()
    check(ctx.lib.sb2_leiden_csr_f32(ctx.handle, n, ptr(d_indptr), ptr(d_indices), ptr(d_weights), float(resolution),
                                     int(n_iterations), int(seed), ptr(member), byref(q), byref(nc), byref(info)))
    return member, q.value, nc.value, dict(passes=info.passes, levels=info.levels, moves=int(info.moves))


def leiden(adj, *, resolution: float = 1.0, n_iterations: int = -1, seed: int = 0, ctx=None):
    """Leiden on a symmetric scipy CSR adjacency -> (membership int32 [n], modularity, info)."""
    ctx = ctx or _abi.default_context()
    adj = adj.tocsr()
    n = adj.shape[0]
    d_indptr, d_indices, d_w = csr_to_device(adj)
    member, q, nc, info = leiden_device(ctx, d_indptr, d_indices, d_w, n, resolution=resolution,
                                        n_iterations=n_iterations, seed=seed)
    info["n_communities"] = nc
    return _to_host(member), q, info


def louvain(adj, *, resolution: float = 1.0, seed: int = 0, ctx=None):
    """Louvain on a symmetric scipy CSR adjacency -> (membership int32 [n], modularity, info)."""
    ctx = ctx or _abi.default_context()
    torch = _torch()
    adj = adj.tocsr()
    n = adj.shape[0]
    d_indptr, d_indices, d_w = csr_to_device(adj)
    member = torch.empty(n, dtype=torch.int32, device="cuda")
    q = c_double()
    nc = c_int32()
    info = LeidenInfo()
    check(ctx.lib.sb2_louvain_csr_f32(ctx.handle, n, ptr(d_indptr), ptr(d_indices), ptr(d_w), float(resolution), int(seed),
                                      ptr(member), byref(q), byref(nc), byref(info)))
    return _to_host(member), q.value, dict(levels=info.levels, moves=int(info.moves), n_communities=nc.value)


def modularity(adj, membership, *, resolution: float = 1.0, ctx=None) -> float:
    ctx = ctx or _abi.default_context()
    adj = adj.tocsr()
    d_indptr, d_indices, d_w = csr_to_device(adj)
    d_m = _to_device(np.asarray(membership, dtype=np.int32))
    q = c_double()
    check(ctx.lib.sb2_modularity_csr_f32(ctx.handle, adj.shape[0], ptr(d_indptr), ptr(d_indices), ptr(d_w),
                                         float(resolution), ptr(d_m), byref(q)))
    return q.value


# ------------------------------------------------------------------------------------------ eigsh / diffmap / umap
def eigsh_scaled_device(ctx, d_indptr, d_indices, d_w, n: int, nev: int, *, d_scale=None, which: str = "LM", v0=None,
                        ncv: int = 0, tol: float = 0.0, max_restarts: int = 0):
    """Extreme eigenpairs of diag(s) A diag(s) on the device -> (evals float64[nev] ascending, evecs CUDA float64 [nev, n], info)."""
    torch = _torch()
    code = {"LA": 0, "LM": 1, "SA": 2}[which]
    if v0 is None:
        v0 = np.random.default_rng(0).standard_normal(n)
    d_v0 = _to_device(np.ascontiguousarray(v0, dtype=np.float64))
    evals = np.empty(nev, np.float64)
    evecs = torch.empty((nev, n), dtype=torch.float64, device="cuda")
    info = EigsInfo()
    check(ctx.lib.sb2_eigsh_csr_scaled(ctx.handle, n, ptr(d_indptr), ptr(d_indices), ptr(d_w),
                                       ptr(d_scale) if d_scale is not None else None, int(nev), code, int(ncv), float(tol),
                                       int(max_restarts), ptr(d_v0), evals.ctypes.data, ptr(evecs), byref(info)))
    return evals, evecs, dict(restarts=info.restarts, matvecs=info.matvecs, n_converged=info.n_converged,
                              max_residual=info.max_residual)


def umap_layout(adj, *, n_components: int, n_epochs: int, a: float, b: float, gamma: float, initial_alpha: float,
                negative_sample_rate: int, seed: int, init, ctx=None):
    """`simplicial_set_embedding` on a symmetric scipy CSR graph -> float32 [n, n_components].
    init: 'spectral' or a float32 [n, n_components] array."""
    torch = _torch()
    ctx = ctx or _abi.default_context()
    adj = adj.tocsr()
    n = adj.shape[0]
    d_indptr, d_indices, d_w = csr_to_device(adj)
    if isinstance(init, str):
        assert init == "spectral"
        emb = torch.empty((n, n_components), dtype=torch.float32, device="cuda")
        check(ctx.lib.sb2_umap_spectral_init_f32(ctx.handle, n, ptr(d_indptr), ptr(d_indices), ptr(d_w), int(n_components),
                                                 int(seed), ptr(emb)))
    else:
        emb = _to_device(np.ascontiguousarray(init, dtype=np.float32))
    check(ctx.lib.sb2_umap_layout_f32(ctx.handle, n, ptr(d_indptr), ptr(d_indices), ptr(d_w), int(n_components), int(n_epochs),
                                      float(a), float(b), float(gamma), float(initial_alpha), int(negative_sample_rate),
                                      int(seed), ptr(emb)))
    return _to_host(emb)


# ------------------------------------------------------------------------------------------ rank_genes_groups
def _csr_f32(x):
    """scipy CSR -> the same matrix with float32 data and canonical (summed duplicate) entries."""
    x = x.tocsr()
    if x.dtype != np.float32:
        x = x.astype(np.float32)
    if not x.has_canonical_format:
        x = x.copy()
        x.sum_duplicates()
    return x


def rank_genes_group_stats(x, codes: np.ndarray, n_codes: int, *, expm1_scale: float = 0.0, ctx=None):
    """Per (code, gene) sums, M2 = sum (x' - mean)^2 and counts of x != 0 over a scipy CSR, x' = expm1(x * expm1_scale)
    (expm1_scale != 0) or x; codes int [n] in 0..n_codes-1.  -> (sum float64, m2 float64, nnz int64), each [n_codes, g]."""
    torch = _torch()
    ctx = ctx or _abi.default_context()
    x = _csr_f32(x)
    n, g = x.shape
    codes = np.asarray(codes, dtype=np.int32)
    rows = np.argsort(codes, kind="stable").astype(np.int32)
    offsets = np.zeros(n_codes + 1, np.int64)
    np.cumsum(np.bincount(codes, minlength=n_codes), out=offsets[1:])
    d_indptr, d_indices, d_data = csr_to_device(x)
    d_rows = _to_device(rows)
    s = torch.empty((n_codes, g), dtype=torch.float64, device="cuda")
    m2 = torch.empty((n_codes, g), dtype=torch.float64, device="cuda")
    nnz = torch.empty((n_codes, g), dtype=torch.int64, device="cuda")
    check(ctx.lib.sb2_rank_genes_group_stats(ctx.handle, n, g, ptr(d_indptr), ptr(d_indices), ptr(d_data), ptr(d_rows),
                                             ptr(offsets), int(n_codes), float(expm1_scale), ptr(s), ptr(m2), ptr(nnz)))
    return _to_host(s, m2, nnz)


def tie_terms_to_int(tie: np.ndarray) -> np.ndarray:
    """(low, high) uint64 halves [..., 2] -> exact Python-int object array [...]."""
    lo, hi = tie[..., 0], tie[..., 1]
    out = np.empty(lo.shape, dtype=object)
    for idx in np.ndindex(lo.shape):
        out[idx] = (int(hi[idx]) << 64) | int(lo[idx])
    return out


def tie_terms_to_f64(tie: np.ndarray) -> np.ndarray:
    """(low, high) uint64 halves [..., 2] -> float64 [...] (the nearest double to within two roundings)."""
    return tie[..., 1].astype(np.float64) * 2.0**64 + tie[..., 0].astype(np.float64)


def rank_genes_wilcoxon(x, codes: np.ndarray, n_codes: int, *, ref: int = -1, stage_ms: list | None = None, ctx=None):
    """Wilcoxon rank sums and tie terms on the device (sb2_rank_genes_wilcoxon); codes int [n] in 0..n_codes-1, code
    n_codes-1 the remainder.  ref < 0: ranks over all cells; else, per code, over that code and `ref` only.
    -> (rank2 int64 [n_codes, g]: twice the rank sums, tie uint64 [n_codes, g, 2]: sum of t^3 - t as low/high halves).
    `stage_ms`, if a list, receives the device milliseconds of the sort and of the rank walk."""
    from ctypes import c_float

    torch = _torch()
    ctx = ctx or _abi.default_context()
    x = _csr_f32(x)
    n, g = x.shape
    codes = np.asarray(codes, dtype=np.int32)
    sizes = np.bincount(codes, minlength=n_codes).astype(np.int64)
    d_indptr, d_indices, d_data = csr_to_device(x)
    d_codes, d_sizes = _to_device(codes), _to_device(sizes)
    rank2 = torch.empty((n_codes, g), dtype=torch.int64, device="cuda")
    tie = torch.empty((n_codes, g, 2), dtype=torch.int64, device="cuda")
    ms = (c_float * 2)() if stage_ms is not None else None
    check(ctx.lib.sb2_rank_genes_wilcoxon(ctx.handle, n, g, ptr(d_indptr), ptr(d_indices), ptr(d_data), int(x.nnz),
                                          ptr(d_codes), ptr(d_sizes), int(n_codes), int(ref), ptr(rank2), ptr(tie),
                                          ms))
    if stage_ms is not None:
        stage_ms[:] = [float(ms[0]), float(ms[1])]
    h_rank2, h_tie = _to_host(rank2, tie)
    return h_rank2, h_tie.view(np.uint64)
