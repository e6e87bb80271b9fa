// rank_genes.cu — the two device reductions behind sc.tl.rank_genes_groups (src/scanpy/tools/_rank_genes_groups.py):
//   sb2_rank_genes_group_stats: per (group, gene) n_g-weighted sum, M2 = sum (x - mean)^2 and count of x != 0 over a CSR,
//     optionally of expm1(x * scale) (`_basic_stats` / `get.aggregate`, :319-452).  Bit-reproducible: every (group, gene)
//     value is a fixed-order sum (warp-private shared-memory accumulators over fixed row chunks, chunks reduced in order).
//   sb2_rank_genes_wilcoxon: doubled Wilcoxon rank sums and exact tie terms sum(t^3 - t) (`wilcoxon`, :505-579) from one
//     stable LSD radix sort of the stored entries on the key (gene | orderable value bits | group code).  After the sort
//     each gene is a segment, each tie run is contiguous and within a run each group's entries are contiguous; the zeros
//     (stored or implicit) form a virtual run between the negative and the positive values.  Integer results only:
//     rank sums accumulate in int64, tie terms in three 32-bit limbs (uint64 accumulators), so atomics are exact and the
//     result does not depend on their order.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------------ grouped statistics
constexpr int ST_WARPS = 4;     // warps per CTA; each warp owns one row chunk and private accumulators
constexpr int ST_TILE = 1024;   // genes per shared-memory tile
constexpr int ST_CHUNK = 2048;  // rows per chunk (all of one group)

__device__ __forceinline__ double transformed(float x, double scale) {
  return scale != 0.0 ? expm1((double)x * scale) : (double)x;
}

// pass 0: part_a[c][j] = sum x', part_n[c][j] = #(x != 0); pass 1: part_a[c][j] = sum_{x != 0} (x' - mean[group][j])^2
template <int PASS>
__global__ void __launch_bounds__(ST_WARPS * 32)
group_stats_kernel(int64_t n_chunks, int32_t g, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                   const float* __restrict__ data, const int32_t* __restrict__ rows, const int64_t* __restrict__ chunk_rows,
                   const int32_t* __restrict__ chunk_group, double scale, const double* __restrict__ mean,
                   double* __restrict__ part_a, int32_t* __restrict__ part_n) {
  extern __shared__ unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* acc = reinterpret_cast<double*>(smem_raw) + warp * ST_TILE;
  int32_t* cnt = reinterpret_cast<int32_t*>(reinterpret_cast<double*>(smem_raw) + ST_WARPS * ST_TILE) + warp * ST_TILE;
  const int64_t c = (int64_t)blockIdx.x * ST_WARPS + warp;
  const int32_t t0 = blockIdx.y * ST_TILE;
  const int32_t tw = min(ST_TILE, g - t0);
  if (c >= n_chunks) return;
  for (int k = lane; k < tw; k += 32) { acc[k] = 0.0; cnt[k] = 0; }
  const double* mu = PASS == 1 ? mean + (size_t)chunk_group[c] * g + t0 : nullptr;
  __syncwarp();
  for (int64_t r = chunk_rows[c]; r < chunk_rows[c + 1]; ++r) {
    const int32_t row = rows[r];
    for (int64_t e = indptr[row] + lane; e < indptr[row + 1]; e += 32) {
      const int32_t k = indices[e] - t0;
      if (k < 0 || k >= tw) continue;
      const float x = data[e];
      if (PASS == 0) {
        acc[k] += transformed(x, scale);
        cnt[k] += x != 0.0f;
      } else if (x != 0.0f) {
        const double d = transformed(x, scale) - mu[k];
        acc[k] += d * d;
      }
    }
    __syncwarp();  // a column appears at most once per row: rows are applied one after another, in chunk order
  }
  for (int k = lane; k < tw; k += 32) {
    part_a[c * g + t0 + k] = acc[k];
    if (PASS == 0) part_n[c * g + t0 + k] = cnt[k];
  }
}

// out[q][j] = chunk partials of group q summed in chunk order; pass 0 also writes nnz and the mean, pass 1 adds the
// implicit zeros' (n_q - nnz) mean^2 to M2
template <int PASS>
__global__ void group_stats_reduce_kernel(int32_t n_codes, int32_t g, const int64_t* __restrict__ group_chunks,
                                          const int64_t* __restrict__ group_rows, const double* __restrict__ part_a,
                                          const int32_t* __restrict__ part_n, double* __restrict__ out_a,
                                          int64_t* __restrict__ out_nnz, double* __restrict__ mean) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_codes * g) return;
  const int32_t q = (int32_t)(i / g), j = (int32_t)(i % g);
  const int64_t nq = group_rows[q + 1] - group_rows[q];
  double s = 0.0;
  int64_t z = 0;
  for (int64_t c = group_chunks[q]; c < group_chunks[q + 1]; ++c) {
    s += part_a[c * g + j];
    if (PASS == 0) z += part_n[c * g + j];
  }
  if (PASS == 0) {
    out_a[i] = s;
    out_nnz[i] = z;
    mean[i] = nq > 0 ? s / (double)nq : 0.0;
  } else {
    const double mu = mean[i];
    out_a[i] = s + (double)(nq - out_nnz[i]) * mu * mu;
  }
}

// ------------------------------------------------------------------------------------------ radix sort
constexpr int RS_WARPS = 8;        // warps per CTA, one tile each
constexpr int RS_TILE = 32 * 256;  // keys per warp tile
constexpr uint32_t ZERO_BITS = 0x80000000u;  // orderable bits of +-0.0f

__device__ __forceinline__ uint32_t orderable(float v) {
  if (v == 0.0f) return ZERO_BITS;
  const uint32_t u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// keys[e] = gene << (32 + gb) | value bits << gb | code[row] for every stored entry (CSR order); or_and[0] |= key,
// or_and[1] &= key (a digit that is equal in both is constant across all keys and its pass can be skipped)
__global__ void __launch_bounds__(256)
build_keys_kernel(int64_t n, const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                  const float* __restrict__ data, const int32_t* __restrict__ codes, int gb, uint64_t* __restrict__ keys,
                  unsigned long long* __restrict__ or_and) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  uint64_t o = 0, a = ~0ull;
  if (row < n) {
    const uint64_t code = (uint64_t)codes[row];
    for (int64_t e = indptr[row] + lane; e < indptr[row + 1]; e += 32) {
      const uint64_t k = ((uint64_t)indices[e] << (32 + gb)) | ((uint64_t)orderable(data[e]) << gb) | code;
      keys[e] = k;
      o |= k;
      a &= k;
    }
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    o |= __shfl_xor_sync(0xffffffffu, o, s);
    a &= __shfl_xor_sync(0xffffffffu, a, s);
  }
  if (lane == 0 && row < n) {
    atomicOr(&or_and[0], (unsigned long long)o);
    atomicAnd(&or_and[1], (unsigned long long)a);
  }
}

// counts[d * n_tiles + tile] = keys of the tile whose digit (key >> shift) & 255 is d
__global__ void __launch_bounds__(RS_WARPS * 32)
radix_hist_kernel(int64_t nnz, const uint64_t* __restrict__ keys, int shift, int64_t n_tiles, int32_t* __restrict__ counts) {
  __shared__ int32_t h[RS_WARPS][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t tile = (int64_t)blockIdx.x * RS_WARPS + warp;
  for (int d = lane; d < 256; d += 32) h[warp][d] = 0;
  __syncwarp();
  if (tile < n_tiles) {
    const int64_t end = min(nnz, (tile + 1) * RS_TILE);
    for (int64_t i = tile * RS_TILE + lane; i < end; i += 32) atomicAdd(&h[warp][(keys[i] >> shift) & 255], 1);
  }
  __syncwarp();
  if (tile < n_tiles)
    for (int d = lane; d < 256; d += 32) counts[(int64_t)d * n_tiles + tile] = h[warp][d];
}

// stable scatter: the tile's keys go, in order, to offsets[d * n_tiles + tile] + (rank among the tile's keys with digit d)
__global__ void __launch_bounds__(RS_WARPS * 32)
radix_scatter_kernel(int64_t nnz, const uint64_t* __restrict__ in, int shift, int64_t n_tiles,
                     const int64_t* __restrict__ offsets, uint64_t* __restrict__ out) {
  __shared__ int64_t base[RS_WARPS][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t tile = (int64_t)blockIdx.x * RS_WARPS + warp;
  if (tile >= n_tiles) return;
  for (int d = lane; d < 256; d += 32) base[warp][d] = offsets[(int64_t)d * n_tiles + tile];
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1u;
  const int64_t end = min(nnz, (tile + 1) * RS_TILE);
  for (int64_t i0 = tile * RS_TILE; i0 < end; i0 += 32) {
    const int64_t i = i0 + lane;
    const bool valid = i < end;
    const uint64_t k = valid ? in[i] : 0;
    const uint32_t d = valid ? (uint32_t)((k >> shift) & 255) : 256u + lane;  // invalid lanes match nobody
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    if (valid) {
      const int64_t b = base[warp][d];
      out[b + __popc(peers & lt)] = k;
      __syncwarp(peers);
      if ((peers & lt) == 0) base[warp][d] = b + __popc(peers);
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------ rank walk
typedef unsigned __int128 u128;

__device__ __forceinline__ u128 tie_term(uint64_t t) { return (u128)t * t * t - t; }

__device__ __forceinline__ void add_limbs(unsigned long long* l, u128 v) {
  if (v == 0) return;
  atomicAdd(l + 0, (unsigned long long)(v & 0xffffffffu));
  atomicAdd(l + 1, (unsigned long long)((v >> 32) & 0xffffffffu));
  atomicAdd(l + 2, (unsigned long long)(v >> 64));
}

__device__ __forceinline__ u128 limbs_value(const unsigned long long* l) {
  return (u128)l[0] + ((u128)l[1] << 32) + ((u128)l[2] << 64);
}

// first x > i (x <= e) with keys[x] >> shift != keys[i] >> shift (galloping: O(log run length) probes)
__device__ int64_t run_end(const uint64_t* __restrict__ k, int64_t i, int64_t e, int shift) {
  const uint64_t r = k[i] >> shift;
  int64_t lo = i, hi = e, step = 1;
  while (true) {
    const int64_t p = lo + step;
    if (p >= e) break;
    if ((k[p] >> shift) != r) { hi = p; break; }
    lo = p;
    step <<= 1;
  }
  while (hi - lo > 1) {
    const int64_t m = lo + (hi - lo) / 2;
    if ((k[m] >> shift) == r) lo = m; else hi = m;
  }
  return hi;
}

// first x >= s with keys[x..i] >> shift all equal to keys[i] >> shift
__device__ int64_t run_begin(const uint64_t* __restrict__ k, int64_t s, int64_t i, int shift) {
  const uint64_t r = k[i] >> shift;
  int64_t lo = s - 1, hi = i, step = 1;
  while (true) {
    const int64_t p = hi - step;
    if (p < s) break;
    if ((k[p] >> shift) != r) { lo = p; break; }
    hi = p;
    step <<= 1;
  }
  while (hi - lo > 1) {
    const int64_t m = lo + (hi - lo) / 2;
    if ((k[m] >> shift) == r) hi = m; else lo = m;
  }
  return hi;
}

// first x in [lo, hi) with keys[x] >= v (hi if none)
__device__ __forceinline__ int64_t lower_bound(const uint64_t* __restrict__ k, int64_t lo, int64_t hi, uint64_t v) {
  while (lo < hi) {
    const int64_t m = lo + (hi - lo) / 2;
    if (k[m] < v) lo = m + 1; else hi = m;
  }
  return lo;
}

__global__ void segments_kernel(int32_t g, int64_t nnz, const uint64_t* __restrict__ keys, int gene_shift,
                                int64_t* __restrict__ seg) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j > g) return;
  seg[j] = j == g ? nnz : lower_bound(keys, 0, nnz, (uint64_t)j << gene_shift);
}

// flags[i] = 1 for a stored non-zero entry of the reference group
__global__ void ref_flags_kernel(int64_t nnz, const uint64_t* __restrict__ keys, int gb, uint64_t ref,
                                 int32_t* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint64_t k = keys[i];
  flags[i] = ((k & ((1ull << gb) - 1)) == ref) && (uint32_t)(k >> gb) != ZERO_BITS;
}

// one thread per sorted entry; the first entry of each (gene, value, group) sub-run of non-zeros does the work.
// Rest mode (ref < 0): every stored entry is ranked; a run of t values starting after C cells has doubled rank
// 2C + t + 1.  Reference mode: U_q doubled, sum over q's entries of 2 #ref below + #ref tied (prefix[] counts the
// reference group's stored non-zeros); cells with code `excl` take no part.
__global__ void __launch_bounds__(256)
rank_walk_kernel(int64_t nnz, int32_t g, int64_t n, const uint64_t* __restrict__ keys, int gb, const int64_t* __restrict__ seg,
                 int32_t ref, int32_t excl, const int64_t* __restrict__ prefix, unsigned long long* __restrict__ rank2,
                 unsigned long long* __restrict__ nz, unsigned long long* __restrict__ neg,
                 unsigned long long* __restrict__ tie, unsigned long long* __restrict__ tie_ref) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint64_t key = keys[i];
  if (i > 0 && keys[i - 1] == key) return;
  const uint32_t vb = (uint32_t)(key >> gb);
  if (vb == ZERO_BITS) return;
  const int32_t q = (int32_t)(key & ((1ull << gb) - 1));
  if (ref >= 0 && q == excl) return;
  const int32_t j = (int32_t)(key >> (32 + gb));
  const int64_t s = seg[j], e = seg[j + 1];
  const int64_t c = run_end(keys, i, e, 0) - i;
  const int64_t a = (i == s || (keys[i - 1] >> gb) != (key >> gb)) ? i : run_begin(keys, s, i, gb);
  const int64_t qj = (int64_t)q * g + j;
  atomicAdd(&nz[qj], (unsigned long long)c);
  if (vb < ZERO_BITS) atomicAdd(&neg[qj], (unsigned long long)c);
  if (ref < 0) {
    const int64_t b = run_end(keys, i + c - 1, e, gb);
    const int64_t t = b - a;
    const int64_t before = (a - s) + (vb > ZERO_BITS ? n - (e - s) : 0);
    atomicAdd(&rank2[qj], (unsigned long long)(c * (2 * before + t + 1)));
    if (i == a) add_limbs(&tie[3 * (int64_t)j], tie_term((uint64_t)t));
    return;
  }
  if (q == ref) {
    add_limbs(&tie_ref[3 * (int64_t)j], tie_term((uint64_t)c));
    return;
  }
  const int64_t b = run_end(keys, i + c - 1, e, gb);
  const uint64_t kref = (key & ~((1ull << gb) - 1)) | (uint64_t)ref;
  const int64_t r0 = lower_bound(keys, a, b, kref);
  const int64_t cref = (r0 < b && keys[r0] == kref) ? run_end(keys, r0, b, 0) - r0 : 0;
  const int64_t below = prefix[a] - prefix[s];
  atomicAdd(&rank2[qj], (unsigned long long)(c * (2 * below + cref)));
  add_limbs(&tie[3 * qj], tie_term((uint64_t)(c + cref)) - tie_term((uint64_t)cref));
}

// adds the zero run and writes the outputs: out_rank2[q][j], out_tie[2 (q g + j) + {0, 1}] = low / high 64 bits
__global__ void rank_finalize_kernel(int32_t n_codes, int32_t g, int64_t n, const uint64_t* __restrict__ keys, int gb,
                                     const int64_t* __restrict__ seg, const int64_t* __restrict__ sizes, int32_t ref,
                                     int32_t excl, const unsigned long long* __restrict__ rank2,
                                     const unsigned long long* __restrict__ nz, const unsigned long long* __restrict__ neg,
                                     const unsigned long long* __restrict__ tie,
                                     const unsigned long long* __restrict__ tie_ref, int64_t* __restrict__ out_rank2,
                                     uint64_t* __restrict__ out_tie) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_codes * g) return;
  const int32_t q = (int32_t)(i / g), j = (int32_t)(i % g);
  const int64_t zq = sizes[q] - (int64_t)nz[i];
  int64_t r2 = 0;
  u128 tt = 0;
  if (ref < 0) {
    const int64_t s = seg[j], e = seg[j + 1];
    const uint64_t gene = (uint64_t)j << (32 + gb);
    const int64_t z0 = lower_bound(keys, s, e, gene | ((uint64_t)ZERO_BITS << gb));
    const int64_t z1 = lower_bound(keys, z0, e, gene | ((uint64_t)(ZERO_BITS + 1) << gb));
    const int64_t n_neg = z0 - s, t0 = n - ((e - s) - (z1 - z0));
    r2 = (int64_t)rank2[i] + zq * (2 * n_neg + t0 + 1);
    tt = limbs_value(&tie[3 * (int64_t)j]) + tie_term((uint64_t)t0);
  } else if (q != ref && q != excl) {
    const int64_t rj = (int64_t)ref * g + j;
    const int64_t zr = sizes[ref] - (int64_t)nz[rj];
    const int64_t nq = sizes[q];
    r2 = (int64_t)rank2[i] + 2 * zr * (int64_t)(nz[i] - neg[i]) + zq * (2 * (int64_t)neg[rj] + zr) + nq * (nq + 1);
    tt = limbs_value(&tie[3 * i]) + limbs_value(&tie_ref[3 * (int64_t)j]) + tie_term((uint64_t)(zq + zr));
  }
  out_rank2[i] = r2;
  out_tie[2 * i] = (uint64_t)tt;
  out_tie[2 * i + 1] = (uint64_t)(tt >> 64);
}

int bits_for(int64_t v) {  // bits needed to hold 0..v
  int b = 0;
  while (b < 63 && (v >> b) != 0) ++b;
  return b;
}

}  // namespace

int32_t sb2_rank_genes_group_stats(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                                   const float* d_data, const int32_t* d_rows, const int64_t* h_group_offsets,
                                   int32_t n_codes, double expm1_scale, double* d_sum, double* d_m2, int64_t* d_nnz) {
  SB2_CHECK_ARG(ctx && n >= 0 && g > 0 && n_codes > 0 && h_group_offsets, "shapes");
  if (n_codes > SB2_RANK_GENES_MAX_GROUPS + 1) {
    sb2_set_error("rank_genes: %d group codes exceed the supported maximum of %d groups (+1 remainder code)", n_codes,
                  SB2_RANK_GENES_MAX_GROUPS);
    return SB2_E_UNSUPPORTED;
  }
  SB2_CHECK_ARG(h_group_offsets[0] == 0 && h_group_offsets[n_codes] == n, "group offsets cover the rows");
  // chunk table: each group's rows (d_rows[offsets[q] : offsets[q + 1]]) split into ST_CHUNK-row chunks
  std::vector<int64_t> chunk_rows{0}, group_chunks{0}, group_rows(h_group_offsets, h_group_offsets + n_codes + 1);
  std::vector<int32_t> chunk_group;
  for (int32_t q = 0; q < n_codes; ++q) {
    SB2_CHECK_ARG(h_group_offsets[q + 1] >= h_group_offsets[q], "group offsets are non-decreasing");
    for (int64_t r = h_group_offsets[q]; r < h_group_offsets[q + 1]; r += ST_CHUNK) {
      chunk_rows.push_back(std::min<int64_t>(r + ST_CHUNK, h_group_offsets[q + 1]));
      chunk_group.push_back(q);
    }
    group_chunks.push_back((int64_t)chunk_group.size());
  }
  const int64_t n_chunks = (int64_t)chunk_group.size();
  ScratchScope scr(ctx);
  int64_t *d_chunk_rows, *d_group_chunks, *d_group_rows;
  int32_t *d_chunk_group, *part_n;
  double *part_a, *mean;
  SB2_TRY(scr.alloc(&d_chunk_rows, chunk_rows.size()));
  SB2_TRY(scr.alloc(&d_group_chunks, group_chunks.size()));
  SB2_TRY(scr.alloc(&d_group_rows, group_rows.size()));
  SB2_TRY(scr.alloc(&d_chunk_group, chunk_group.size()));
  SB2_TRY(scr.alloc(&part_a, (size_t)n_chunks * g));
  SB2_TRY(scr.alloc(&part_n, (size_t)n_chunks * g));
  SB2_TRY(scr.alloc(&mean, (size_t)n_codes * g));
  SB2_CUDA(cudaMemcpyAsync(d_chunk_rows, chunk_rows.data(), chunk_rows.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  SB2_CUDA(cudaMemcpyAsync(d_group_chunks, group_chunks.data(), group_chunks.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  SB2_CUDA(cudaMemcpyAsync(d_group_rows, group_rows.data(), group_rows.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  if (n_chunks > 0)
    SB2_CUDA(cudaMemcpyAsync(d_chunk_group, chunk_group.data(), chunk_group.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  const size_t smem = (size_t)ST_WARPS * ST_TILE * (sizeof(double) + sizeof(int32_t));
  const dim3 grid((unsigned)std::max<int64_t>(1, ceil_div64(n_chunks, ST_WARPS)), (unsigned)ceil_div64(g, ST_TILE));
  const int64_t cells = (int64_t)n_codes * g;
  const unsigned rgrid = (unsigned)ceil_div64(cells, 256);
  if (n_chunks > 0) {
    group_stats_kernel<0><<<grid, ST_WARPS * 32, smem, ctx->stream>>>(n_chunks, g, d_indptr, d_indices, d_data, d_rows,
                                                                       d_chunk_rows, d_chunk_group, expm1_scale, nullptr,
                                                                       part_a, part_n);
    SB2_LAUNCH_CHECK(ctx);
  }
  group_stats_reduce_kernel<0><<<rgrid, 256, 0, ctx->stream>>>(n_codes, g, d_group_chunks, d_group_rows, part_a, part_n,
                                                                d_sum, d_nnz, mean);
  SB2_LAUNCH_CHECK(ctx);
  if (n_chunks > 0) {
    group_stats_kernel<1><<<grid, ST_WARPS * 32, smem, ctx->stream>>>(n_chunks, g, d_indptr, d_indices, d_data, d_rows,
                                                                       d_chunk_rows, d_chunk_group, expm1_scale, mean,
                                                                       part_a, part_n);
    SB2_LAUNCH_CHECK(ctx);
  }
  group_stats_reduce_kernel<1><<<rgrid, 256, 0, ctx->stream>>>(n_codes, g, d_group_chunks, d_group_rows, part_a, part_n,
                                                                d_m2, d_nnz, mean);
  SB2_LAUNCH_CHECK(ctx);
  return SB2_OK;
}

int32_t sb2_rank_genes_wilcoxon(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                                const float* d_data, int64_t nnz, const int32_t* d_codes, const int64_t* d_group_sizes,
                                int32_t n_codes, int32_t ref, int64_t* d_rank2, uint64_t* d_tie, float* h_stage_ms) {
  SB2_CHECK_ARG(ctx && n >= 0 && g > 0 && nnz >= 0 && n_codes > 0 && ref < n_codes - 1, "shapes");
  if (n_codes > SB2_RANK_GENES_MAX_GROUPS + 1) {
    sb2_set_error("rank_genes: %d group codes exceed the supported maximum of %d groups (+1 remainder code)", n_codes,
                  SB2_RANK_GENES_MAX_GROUPS);
    return SB2_E_UNSUPPORTED;
  }
  const int gb = std::max(1, bits_for(n_codes - 1));
  const int gene_shift = 32 + gb;
  if (bits_for(g) + gene_shift > 64) {
    sb2_set_error("rank_genes: %d genes x %d group codes do not fit the 64-bit sort key", g, n_codes);
    return SB2_E_UNSUPPORTED;
  }
  const bool ref_mode = ref >= 0;
  const int32_t excl = n_codes - 1;
  ScratchScope scr(ctx);
  uint64_t *keys, *alt;
  unsigned long long *or_and, *rank2, *nz, *neg, *tie, *tie_ref;
  int64_t *seg, *prefix = nullptr;
  const int64_t cells = (int64_t)n_codes * g;
  const int64_t tie_len = ref_mode ? 3 * cells : 3 * (int64_t)g;
  SB2_TRY(scr.alloc(&keys, (size_t)nnz));
  SB2_TRY(scr.alloc(&alt, (size_t)nnz));
  SB2_TRY(scr.alloc(&or_and, 2));
  SB2_TRY(scr.alloc(&seg, (size_t)g + 1));
  SB2_TRY(scr.alloc(&rank2, (size_t)cells));
  SB2_TRY(scr.alloc(&nz, (size_t)cells));
  SB2_TRY(scr.alloc(&neg, (size_t)cells));
  SB2_TRY(scr.alloc(&tie, (size_t)tie_len));
  SB2_TRY(scr.alloc(&tie_ref, 3 * (size_t)g));
  SB2_CUDA(cudaMemsetAsync(or_and, 0, 8, ctx->stream));
  SB2_CUDA(cudaMemsetAsync(or_and + 1, 0xff, 8, ctx->stream));
  SB2_CUDA(cudaMemsetAsync(rank2, 0, cells * 8, ctx->stream));
  SB2_CUDA(cudaMemsetAsync(nz, 0, cells * 8, ctx->stream));
  SB2_CUDA(cudaMemsetAsync(neg, 0, cells * 8, ctx->stream));
  SB2_CUDA(cudaMemsetAsync(tie, 0, tie_len * 8, ctx->stream));
  SB2_CUDA(cudaMemsetAsync(tie_ref, 0, 3 * (size_t)g * 8, ctx->stream));
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  if (h_stage_ms) {
    for (auto& e : ev) SB2_CUDA(cudaEventCreate(&e));
    SB2_CUDA(cudaEventRecord(ev[0], ctx->stream));
  }
  if (nnz > 0) {
    build_keys_kernel<<<(unsigned)ceil_div64(std::max<int64_t>(n, 1), 8), 256, 0, ctx->stream>>>(
        n, d_indptr, d_indices, d_data, d_codes, gb, keys, or_and);
    SB2_LAUNCH_CHECK(ctx);
    unsigned long long h_or_and[2];
    SB2_CUDA(cudaMemcpyAsync(h_or_and, or_and, 16, cudaMemcpyDeviceToHost, ctx->stream));
    SB2_CUDA(cudaStreamSynchronize(ctx->stream));
    const uint64_t varying = h_or_and[0] ^ h_or_and[1];
    const int64_t n_tiles = ceil_div64(nnz, RS_TILE);
    int32_t* counts;
    int64_t* offsets;
    SB2_TRY(scr.alloc(&counts, (size_t)n_tiles * 256));
    SB2_TRY(scr.alloc(&offsets, (size_t)n_tiles * 256 + 1));
    const unsigned rs_grid = (unsigned)ceil_div64(n_tiles, RS_WARPS);
    for (int shift = 0; shift < 64; shift += 8) {
      if (((varying >> shift) & 255) == 0) continue;  // every key has the same digit here: the pass is the identity
      radix_hist_kernel<<<rs_grid, RS_WARPS * 32, 0, ctx->stream>>>(nnz, keys, shift, n_tiles, counts);
      SB2_LAUNCH_CHECK(ctx);
      SB2_TRY(sb2_scan_i32_to_i64(ctx, counts, n_tiles * 256, offsets));
      radix_scatter_kernel<<<rs_grid, RS_WARPS * 32, 0, ctx->stream>>>(nnz, keys, shift, n_tiles, offsets, alt);
      SB2_LAUNCH_CHECK(ctx);
      std::swap(keys, alt);
    }
  }
  if (h_stage_ms) SB2_CUDA(cudaEventRecord(ev[1], ctx->stream));
  segments_kernel<<<(unsigned)ceil_div64((int64_t)g + 1, 256), 256, 0, ctx->stream>>>(g, nnz, keys, gene_shift, seg);
  SB2_LAUNCH_CHECK(ctx);
  if (ref_mode && nnz > 0) {
    int32_t* flags;
    SB2_TRY(scr.alloc(&flags, (size_t)nnz));
    SB2_TRY(scr.alloc(&prefix, (size_t)nnz + 1));
    ref_flags_kernel<<<(unsigned)ceil_div64(nnz, 256), 256, 0, ctx->stream>>>(nnz, keys, gb, (uint64_t)ref, flags);
    SB2_LAUNCH_CHECK(ctx);
    SB2_TRY(sb2_scan_i32_to_i64(ctx, flags, nnz, prefix));
  }
  if (nnz > 0) {
    rank_walk_kernel<<<(unsigned)ceil_div64(nnz, 256), 256, 0, ctx->stream>>>(nnz, g, n, keys, gb, seg, ref, excl, prefix,
                                                                             rank2, nz, neg, tie, tie_ref);
    SB2_LAUNCH_CHECK(ctx);
  }
  rank_finalize_kernel<<<(unsigned)ceil_div64(cells, 256), 256, 0, ctx->stream>>>(
      n_codes, g, n, keys, gb, seg, d_group_sizes, ref, excl, rank2, nz, neg, tie, tie_ref, d_rank2, d_tie);
  SB2_LAUNCH_CHECK(ctx);
  if (h_stage_ms) {
    SB2_CUDA(cudaEventRecord(ev[2], ctx->stream));
    SB2_CUDA(cudaEventSynchronize(ev[2]));
    SB2_CUDA(cudaEventElapsedTime(&h_stage_ms[0], ev[0], ev[1]));
    SB2_CUDA(cudaEventElapsedTime(&h_stage_ms[1], ev[1], ev[2]));
    for (auto& e : ev) cudaEventDestroy(e);
  }
  return SB2_OK;
}
