// rulebook.cu -- sparse-convolution rulebooks as dense neighbour tables (b2s_hash_build,
// b2s_rulebook_subm, b2s_rulebook_conv, b2s_rulebook_pairs; see include/b2second.h).
//
// Instead of spconv's per-offset pair lists (gather / GEMM / scatter-add per offset, one D2H sync per
// layer) the rulebook is OUTPUT-STATIONARY: nbr[o][k] = input row feeding output row o through kernel
// offset k (or -1).  A conv is then one pass with one write per output row and no atomics.
//   cross-correlation: out[o] = sum_k W[k]^T in[o*s - p + k*d],  k row-major over (kz,ky,kx).
//
// Strided conv output set: {o : exists k, o*s - p + k*d is active}, emitted sorted ascending by flat
// (b,z,y,x) key (the order upstream's GPU path produces with thrust sort+unique).  Here dedup + sort
// are one step: an occupancy bitmap over the output grid plus a popcount prefix scan gives every
// active output cell its sorted rank directly.
//
// The occupancy structure is two-level (round 2): a summary bitmap (one bit per 32-cell word) is set by the marking
// pass, so ranking and emitting touch only the NON-EMPTY words (a few hundred thousand) instead of scanning the whole
// output grid (21 x 800 x 704 x 32 frames = 11.8 M words at the first strided conv of car.fhd: k_popc_scan +
// k_conv_emit cost 138 us per step there, ncu launch list).  Every non-empty word w also records the output row of
// its first cell, wrow0[w]; coordinate -> row is then `bit set ? wrow0[w] + popc(bits below) : none` -- two loads, no
// probing -- which b2s_rulebook_subm_ranked uses for the SubM table of the level a strided conv has just produced
// (no hash table for that level at all).
//
// All row counts are read from device memory; grids are bounded (a few CTAs per SM) with grid-stride loops,
// so the cost follows the live row count, not the buffer capacity (capacity-sized grids cost ~40 us per
// launch of mostly-idle threads in the first profile).
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kScanThreads = 1024;
constexpr int kMaxBlocks = 148 * 8;

inline int bounded_grid(long long work_items, int threads)
{
    long long b = (work_items + threads - 1) / threads;
    if (b < 1) b = 1;
    return (int)(b < kMaxBlocks ? b : kMaxBlocks);
}

struct ConvGeom {
    int in_shape[3], out_shape[3], k[3], s[3], p[3], d[3];
    int K;
};

__global__ void k_hash_build(const int *__restrict__ coors, const int *__restrict__ n_dev, int cap_rows,
                             int D, int H, int W, unsigned long long *keys, int *vals, int mask,
                             unsigned *status)
{
    const int n = min(*n_dev, cap_rows);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int4 c = *reinterpret_cast<const int4 *>(coors + (size_t)i * 4);
        unsigned long long key = b2s_flat_key(c.x, c.y, c.z, c.w, D, H, W);
        int h = b2s_hash_insert(keys, mask, key);
        if (h < 0) { atomicOr(status, B2S_STATUS_HASH_FULL); continue; }
        vals[h] = i;
    }
}

// SubM neighbour table.  The relation is symmetric (j = i + delta  <=>  i = j - delta, mirrored offset index
// K-1-k), so only the first half of the offsets is looked up and both entries are written; nbr is pre-filled
// with -1 by the caller.  One thread per (row, k < K/2).
__global__ void k_subm_nbr(const int *__restrict__ coors, const int *__restrict__ n_dev, int cap_rows,
                           ConvGeom g, const unsigned long long *__restrict__ keys,
                           const int *__restrict__ vals, int mask, int *nbr, unsigned *row_mask)
{
    const int n = min(*n_dev, cap_rows);
    const int half = g.K / 2;            // offsets 0..half-1 are looked up, `half` is the centre
    const long long total = (long long)n * (half + 1);
    for (long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x; gid < total;
         gid += (long long)gridDim.x * blockDim.x) {
        int row = (int)(gid / (half + 1)), k = (int)(gid % (half + 1));
        if (k == half) {
            nbr[(size_t)row * g.K + half] = row;
            if (row_mask) atomicOr(&row_mask[row], 1u << half);
            continue;
        }
        int kx = k % g.k[2], ky = (k / g.k[2]) % g.k[1], kz = k / (g.k[2] * g.k[1]);
        int4 c = *reinterpret_cast<const int4 *>(coors + (size_t)row * 4);
        int z = c.y + (kz - g.k[0] / 2) * g.d[0];
        int y = c.z + (ky - g.k[1] / 2) * g.d[1];
        int x = c.w + (kx - g.k[2] / 2) * g.d[2];
        if (z < 0 || z >= g.in_shape[0] || y < 0 || y >= g.in_shape[1] || x < 0 || x >= g.in_shape[2]) continue;
        int j = b2s_hash_find(keys, vals, mask,
                              b2s_flat_key(c.x, z, y, x, g.in_shape[0], g.in_shape[1], g.in_shape[2]));
        if (j >= 0 && j < n) {
            nbr[(size_t)row * g.K + k] = j;
            nbr[(size_t)j * g.K + (g.K - 1 - k)] = row;
            if (row_mask) {                      // which offsets each row has (input of b2s_sparse_tile_plan)
                atomicOr(&row_mask[row], 1u << k);
                atomicOr(&row_mask[j], 1u << (g.K - 1 - k));
            }
        }
    }
}

// one thread per input row: mark every output cell the row contributes to
__global__ void k_conv_mark(const int *__restrict__ coors, const int *__restrict__ n_dev, int cap_rows,
                            ConvGeom g, unsigned *bitmap, unsigned *summary)
{
    const int n = min(*n_dev, cap_rows);
    for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < n; row += gridDim.x * blockDim.x) {
        int4 c = *reinterpret_cast<const int4 *>(coors + (size_t)row * 4);
        const int ic[3] = {c.y, c.z, c.w};
        // per dimension: the (<= ceil(k/s)) valid output coordinates
        int oc[3][4], cnt[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            cnt[j] = 0;
            for (int kk = 0; kk < g.k[j]; ++kk) {
                int num = ic[j] + g.p[j] - kk * g.d[j];
                if (num < 0 || num % g.s[j] != 0) continue;
                int o = num / g.s[j];
                if (o >= g.out_shape[j]) continue;
                bool dup = false;
                for (int q = 0; q < cnt[j]; ++q) dup |= (oc[j][q] == o);
                if (!dup && cnt[j] < 4) oc[j][cnt[j]++] = o;
            }
        }
        for (int a = 0; a < cnt[0]; ++a)
            for (int b = 0; b < cnt[1]; ++b)
                for (int e = 0; e < cnt[2]; ++e) {
                    unsigned long long key = b2s_flat_key(c.x, oc[0][a], oc[1][b], oc[2][e], g.out_shape[0],
                                                          g.out_shape[1], g.out_shape[2]);
                    unsigned bit = 1u << (key & 31);
                    const unsigned long long wi = key >> 5;
                    unsigned *w = &bitmap[wi];
                    if (!(*(volatile unsigned *)w & bit)) {
                        // exactly one thread sees the word go from empty to non-empty: it sets the summary bit
                        if (atomicOr(w, bit) == 0u) atomicOr(&summary[wi >> 5], 1u << (wi & 31));
                    }
                }
    }
}

// level 1: exclusive scan of popc(summary word) -> rank of the first non-empty bitmap word below each summary word
__global__ void k_summary_scan(const unsigned *__restrict__ summary, long long nsw, int *sum_prefix, int *block_sums)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int v = i < nsw ? __popc(summary[i]) : 0;
    int total;
    int ex = b2s_block_exscan(v, &total);
    if (i < nsw) sum_prefix[i] = ex;
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single-block exclusive scan of per-block sums; nblk from the host, or (nblk_dev) ceil(*nblk_dev / kScanThreads).
// total -> *total_dev (clamped to cap, raising the overflow flag, when status is given)
__global__ void k_scan_sums(int *block_sums, int nblk_host, const int *items_dev, int *total_dev, int cap,
                            unsigned *status)
{
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int nblk = items_dev ? (*items_dev + kScanThreads - 1) / kScanThreads : nblk_host;
    for (int base = 0; base < nblk; base += blockDim.x) {
        int idx = base + threadIdx.x;
        int v = idx < nblk ? block_sums[idx] : 0;
        int total;
        int ex = b2s_block_exscan(v, &total);
        int c = carry;
        if (idx < nblk) block_sums[idx] = c + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry = c + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int n = carry;
        if (status && n > cap) { atomicOr(status, B2S_STATUS_ROWS_OVERFLOW); n = cap; }
        *total_dev = n;
    }
}

// compact the non-empty bitmap words: nz_word[r] = word index, nz_cnt[r] = its popcount (r ascending in word index)
__global__ void k_compact_words(const unsigned *__restrict__ summary, long long nsw, const int *__restrict__ sum_prefix,
                                const int *__restrict__ block_prefix, const unsigned *__restrict__ bitmap, int *nz_word,
                                int *nz_cnt)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nsw; i += (long long)gridDim.x * blockDim.x) {
        unsigned sbits = summary[i];
        if (!sbits) continue;
        int r = block_prefix[i / kScanThreads] + sum_prefix[i];
        while (sbits) {
            const int j = __ffs(sbits) - 1;
            sbits &= sbits - 1;
            const long long w = i * 32 + j;
            nz_word[r] = (int)w;
            nz_cnt[r] = __popc(bitmap[w]);
            ++r;
        }
    }
}

// level 2: exclusive scan of the non-empty words' popcounts in chunks of kScanThreads (bounded grid, chunk-stride)
__global__ void k_nz_scan(int *nz_cnt /*in: counts, out: exclusive prefix inside the chunk*/, const int *__restrict__ nnz_dev,
                          int *chunk_sums)
{
    const int nnz = *nnz_dev;
    for (long long base = (long long)blockIdx.x * kScanThreads; base < nnz; base += (long long)gridDim.x * kScanThreads) {
        const long long i = base + threadIdx.x;
        int v = i < nnz ? nz_cnt[i] : 0;
        int total;
        int ex = b2s_block_exscan(v, &total);
        if (i < nnz) nz_cnt[i] = ex;
        if (threadIdx.x == 0) chunk_sums[base / kScanThreads] = total;
    }
}

// warp per 32 non-empty words; the bits of each word are expanded by the 32 lanes in parallel.  Writes the output
// coordinates (ascending flat key = the order upstream's sort + unique produces), wrow0[word] = first row of the word,
// and pre-fills the rows' neighbour-table entries with -1.
__global__ void k_conv_emit(const unsigned *__restrict__ bitmap, const int *__restrict__ nz_word,
                            const int *__restrict__ nz_prefix, const int *__restrict__ chunk_prefix,
                            const int *__restrict__ nnz_dev, ConvGeom g, int cap_out, int *coors_out, int *nbr_fill,
                            int *wrow0)
{
    const int lane = threadIdx.x & 31;
    const long long warps_total = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned W = g.out_shape[2], H = g.out_shape[1], D = g.out_shape[0];
    const int nnz = *nnz_dev;
    for (long long base = warp0 * 32; base < nnz; base += warps_total * 32) {
        const long long i = base + lane;
        const int my_word = i < nnz ? nz_word[i] : 0;
        const unsigned bits = i < nnz ? bitmap[my_word] : 0u;
        const int my_row0 = i < nnz ? chunk_prefix[i / kScanThreads] + nz_prefix[i] : 0;
        if (i < nnz) wrow0[my_word] = my_row0;
        const int cnt_here = (int)min((long long)32, (long long)nnz - base);
        for (int src = 0; src < cnt_here; ++src) {
            const unsigned wbits = __shfl_sync(0xffffffffu, bits, src);
            const int row0 = __shfl_sync(0xffffffffu, my_row0, src);
            const int word = __shfl_sync(0xffffffffu, my_word, src);
            if (nbr_fill) {
                // the rows of one bitmap word are consecutive: pre-fill their neighbour-table entries with -1
                // (coalesced) for k_conv_scatter_nbr, instead of a capacity-sized memset
                const int cnt = min(__popc(wbits), max(cap_out - row0, 0));
                for (int q = lane; q < cnt * g.K; q += 32) nbr_fill[(size_t)row0 * g.K + q] = -1;
            }
            if (wbits & (1u << lane)) {
                int row = row0 + __popc(wbits & ((1u << lane) - 1u));
                if (row < cap_out) {
                    unsigned long long key = (((unsigned long long)(unsigned)word) << 5) + lane;
                    unsigned long long r = key / W;
                    int x = (int)(key - r * W);
                    unsigned long long r2 = r / H;
                    int y = (int)(r - r2 * H);
                    int b = (int)(r2 / D);
                    int z = (int)(r2 - (unsigned long long)b * D);
                    *reinterpret_cast<int4 *>(coors_out + (size_t)row * 4) = make_int4(b, z, y, x);
                }
            }
        }
    }
}

// one thread per (output row, k): neighbour lookup in the input hash
__global__ void k_conv_nbr(const int *__restrict__ coors_out, const int *__restrict__ n_out_dev, int cap_out,
                           ConvGeom g, const unsigned long long *__restrict__ keys_in,
                           const int *__restrict__ vals_in, int mask_in, int *nbr, unsigned *row_mask)
{
    const int n = min(*n_out_dev, cap_out);
    const long long total = (long long)n * g.K;
    for (long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x; gid < total;
         gid += (long long)gridDim.x * blockDim.x) {
        int row = (int)(gid / g.K), k = (int)(gid % g.K);
        int kk[3] = {k / (g.k[2] * g.k[1]), (k / g.k[2]) % g.k[1], k % g.k[2]};
        int4 c = *reinterpret_cast<const int4 *>(coors_out + (size_t)row * 4);
        int oc[3] = {c.y, c.z, c.w};
        int ic[3];
        bool ok = true;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            ic[j] = oc[j] * g.s[j] - g.p[j] + kk[j] * g.d[j];
            if (ic[j] < 0 || ic[j] >= g.in_shape[j]) ok = false;
        }
        int r = -1;
        if (ok)
            r = b2s_hash_find(keys_in, vals_in, mask_in,
                              b2s_flat_key(c.x, ic[0], ic[1], ic[2], g.in_shape[0], g.in_shape[1], g.in_shape[2]));
        nbr[gid] = r;
        if (row_mask && r >= 0) atomicOr(&row_mask[row], 1u << k);
    }
}

// The same table built from the INPUT side: every input row visits the (<= ceil(k/s)^3) output cells it feeds,
// ranks each cell in the occupancy bitmap (block prefix + word prefix + popcount of the lower bits = its output
// row, exactly what k_conv_emit assigns) and writes nbr[row_out][k] = row_in.  Work is proportional to the
// (input, output) pairs instead of rows_out * K hash probes of which ~70 % miss (k_conv_nbr: 36 us vs the
// level's 14 us mark pass, ncu launch list round 1); nbr is pre-filled with -1 by the caller.
__global__ void k_conv_scatter_nbr(const int *__restrict__ coors_in, const int *__restrict__ n_in_dev, int cap_in,
                                   ConvGeom g, const unsigned *__restrict__ bitmap,
                                   const int *__restrict__ wrow0, int cap_out, int *nbr, unsigned *row_mask)
{
    const int n = min(*n_in_dev, cap_in);
    for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < n; row += gridDim.x * blockDim.x) {
        int4 c = *reinterpret_cast<const int4 *>(coors_in + (size_t)row * 4);
        const int ic[3] = {c.y, c.z, c.w};
        int oc[3][4], okk[3][4], cnt[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            cnt[j] = 0;
            for (int kk = 0; kk < g.k[j]; ++kk) {
                int num = ic[j] + g.p[j] - kk * g.d[j];
                if (num < 0 || num % g.s[j] != 0) continue;
                int o = num / g.s[j];
                if (o >= g.out_shape[j] || cnt[j] >= 4) continue;
                oc[j][cnt[j]] = o;
                okk[j][cnt[j]] = kk;
                ++cnt[j];
            }
        }
        for (int a = 0; a < cnt[0]; ++a)
            for (int b = 0; b < cnt[1]; ++b)
                for (int e = 0; e < cnt[2]; ++e) {
                    const unsigned long long key = b2s_flat_key(c.x, oc[0][a], oc[1][b], oc[2][e], g.out_shape[0],
                                                                g.out_shape[1], g.out_shape[2]);
                    const long long w = (long long)(key >> 5);
                    const unsigned bit = (unsigned)(key & 31);
                    const int row_out = wrow0[w] + __popc(bitmap[w] & ((1u << bit) - 1u));
                    const int k = (okk[0][a] * g.k[1] + okk[1][b]) * g.k[2] + okk[2][e];
                    if (row_out < cap_out) {
                        nbr[(size_t)row_out * g.K + k] = row;
                        if (row_mask) atomicOr(&row_mask[row_out], 1u << k);
                    }
                }
    }
}

// SubM neighbour table of a level whose occupancy structure (bitmap + wrow0, from the strided conv that produced it)
// is still in the workspace: coordinate -> row is a bit test + rank, no hash probing.  Symmetric like k_subm_nbr: one
// thread per (row, k < K/2) writes both directions.
__global__ void k_subm_ranked(const int *__restrict__ coors, const int *__restrict__ n_dev, int cap_rows, ConvGeom g,
                              const unsigned *__restrict__ bitmap, const int *__restrict__ wrow0, int *nbr,
                              unsigned *row_mask)
{
    const int n = min(*n_dev, cap_rows);
    const int half = g.K / 2;
    const long long total = (long long)n * (half + 1);
    for (long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x; gid < total;
         gid += (long long)gridDim.x * blockDim.x) {
        int row = (int)(gid / (half + 1)), k = (int)(gid % (half + 1));
        if (k == half) {
            nbr[(size_t)row * g.K + half] = row;
            if (row_mask) atomicOr(&row_mask[row], 1u << half);
            continue;
        }
        int kx = k % g.k[2], ky = (k / g.k[2]) % g.k[1], kz = k / (g.k[2] * g.k[1]);
        int4 c = *reinterpret_cast<const int4 *>(coors + (size_t)row * 4);
        int z = c.y + (kz - g.k[0] / 2) * g.d[0];
        int y = c.z + (ky - g.k[1] / 2) * g.d[1];
        int x = c.w + (kx - g.k[2] / 2) * g.d[2];
        if (z < 0 || z >= g.in_shape[0] || y < 0 || y >= g.in_shape[1] || x < 0 || x >= g.in_shape[2]) continue;
        const unsigned long long key = b2s_flat_key(c.x, z, y, x, g.in_shape[0], g.in_shape[1], g.in_shape[2]);
        const unsigned bits = __ldg(&bitmap[key >> 5]);
        const unsigned bit = (unsigned)(key & 31);
        if (!((bits >> bit) & 1u)) continue;
        const int j = __ldg(&wrow0[key >> 5]) + __popc(bits & ((1u << bit) - 1u));
        if (j < n) {
            nbr[(size_t)row * g.K + k] = j;
            nbr[(size_t)j * g.K + (g.K - 1 - k)] = row;
            if (row_mask) {
                atomicOr(&row_mask[row], 1u << k);
                atomicOr(&row_mask[j], 1u << (g.K - 1 - k));
            }
        }
    }
}

__global__ void k_pairs(const int *__restrict__ nbr, const int *__restrict__ n_out_dev, int cap_out, int K,
                        int L, int *pairs, int *pair_num)
{
    const int n = min(*n_out_dev, cap_out);
    const long long total = (long long)n * K;
    for (long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x; gid < total;
         gid += (long long)gridDim.x * blockDim.x) {
        int row = (int)(gid / K), k = (int)(gid % K);
        int r = nbr[gid];
        if (r < 0) continue;
        int pos = atomicAdd(&pair_num[k], 1);
        if (pos < L) {
            pairs[((size_t)k * 2 + 0) * L + pos] = r;
            pairs[((size_t)k * 2 + 1) * L + pos] = row;
        }
    }
}

struct ConvWorkspace {
    unsigned *bitmap, *summary;
    int *sum_prefix, *sum_blocks, *nnz, *nz_word, *nz_prefix, *chunk_sums, *wrow0;
    long long nwords, nsw;
    int nblk_s, nchunks;
};

size_t carve(ConvWorkspace *w, char *base, int batch, const int *out_shape)
{
    long long cells = (long long)batch * out_shape[0] * out_shape[1] * out_shape[2];
    long long nwords = (cells + 31) / 32;
    long long nsw = (nwords + 31) / 32;
    int nblk_s = b2s_cdiv(nsw > 0 ? nsw : 1, kScanThreads);
    int nchunks = b2s_cdiv(nwords > 0 ? nwords : 1, kScanThreads);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += b2s_align(bytes); return base ? base + o : nullptr; };
    // bitmap and summary are contiguous: one memset clears both
    unsigned *bitmap = (unsigned *)take(sizeof(unsigned) * (size_t)(nwords + nsw));
    int *sp = (int *)take(sizeof(int) * (size_t)nsw);
    int *sb = (int *)take(sizeof(int) * (size_t)(nblk_s + 1));
    int *nnz = (int *)take(sizeof(int) * 4);
    int *nzw = (int *)take(sizeof(int) * (size_t)nwords);
    int *nzp = (int *)take(sizeof(int) * (size_t)nwords);
    int *cs = (int *)take(sizeof(int) * (size_t)(nchunks + 1));
    int *wr = (int *)take(sizeof(int) * (size_t)nwords);
    if (w) {
        w->bitmap = bitmap; w->summary = bitmap ? bitmap + nwords : nullptr; w->sum_prefix = sp; w->sum_blocks = sb;
        w->nnz = nnz; w->nz_word = nzw; w->nz_prefix = nzp; w->chunk_sums = cs; w->wrow0 = wr;
        w->nwords = nwords; w->nsw = nsw; w->nblk_s = nblk_s; w->nchunks = nchunks;
    }
    return off;
}

int fill_geom(ConvGeom *g, const int *in_shape, const int *out_shape, const int *ksize, const int *stride,
              const int *padding, const int *dilation)
{
    for (int j = 0; j < 3; ++j) {
        g->in_shape[j] = in_shape[j];
        g->out_shape[j] = out_shape ? out_shape[j] : in_shape[j];
        g->k[j] = ksize[j];
        g->s[j] = stride ? stride[j] : 1;
        g->p[j] = padding ? padding[j] : 0;
        g->d[j] = dilation ? dilation[j] : 1;
        if (g->k[j] < 1 || g->s[j] < 1 || g->d[j] < 1 || g->in_shape[j] < 1 || g->out_shape[j] < 1) return -1;
    }
    g->K = g->k[0] * g->k[1] * g->k[2];
    return 0;
}

}  // namespace

extern "C" int b2s_hash_build(const int *coors, const int *num_rows_dev, int cap_rows, const int *shape,
                              unsigned long long *hash_keys, int *hash_vals, int hash_cap,
                              unsigned *status_dev, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    B2S_REQUIRE((hash_cap & (hash_cap - 1)) == 0 && hash_cap >= 2 * cap_rows && hash_cap >= 2,
                "b2s_hash_build: hash_cap must be a power of two >= 2*cap_rows");
    B2S_CUDA_OK(cudaMemsetAsync(hash_keys, 0xFF, sizeof(unsigned long long) * (size_t)hash_cap, stream));
    B2S_CUDA_OK(cudaMemsetAsync(hash_vals, 0xFF, sizeof(int) * (size_t)hash_cap, stream));
    if (cap_rows > 0) {
        k_hash_build<<<bounded_grid(cap_rows, kThreads), kThreads, 0, stream>>>(
            coors, num_rows_dev, cap_rows, shape[0], shape[1], shape[2], hash_keys, hash_vals, hash_cap - 1,
            status_dev);
        B2S_LAUNCH_OK();
    }
    return 0;
}

extern "C" int b2s_rulebook_subm(const int *coors, const int *num_rows_dev, int cap_rows, const int *shape,
                                 const int *ksize, const int *dilation, const unsigned long long *hash_keys,
                                 const int *hash_vals, int hash_cap, int *nbr, unsigned *row_mask, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    ConvGeom g;
    B2S_REQUIRE(fill_geom(&g, shape, nullptr, ksize, nullptr, nullptr, dilation) == 0,
                "b2s_rulebook_subm: bad geometry");
    B2S_REQUIRE((g.k[0] & 1) && (g.k[1] & 1) && (g.k[2] & 1), "b2s_rulebook_subm: kernel sizes must be odd");
    if (cap_rows > 0) {
        B2S_CUDA_OK(cudaMemsetAsync(nbr, 0xFF, sizeof(int) * (size_t)cap_rows * g.K, stream));
        if (row_mask) B2S_CUDA_OK(cudaMemsetAsync(row_mask, 0, sizeof(unsigned) * (size_t)cap_rows, stream));
        k_subm_nbr<<<bounded_grid((long long)cap_rows * (g.K / 2 + 1), kThreads), kThreads, 0, stream>>>(
            coors, num_rows_dev, cap_rows, g, hash_keys, hash_vals, hash_cap - 1, nbr, row_mask);
        B2S_LAUNCH_OK();
    }
    return 0;
}

extern "C" size_t b2s_rulebook_conv_workspace_bytes(int batch, const int *out_shape)
{
    return carve(nullptr, nullptr, batch, out_shape);
}

extern "C" int b2s_rulebook_conv(const int *coors_in, const int *num_in_dev, int cap_in, int batch,
                                 const int *in_shape, const int *out_shape, const int *ksize,
                                 const int *stride, const int *padding, const int *dilation,
                                 const unsigned long long *hash_keys_in, const int *hash_vals_in,
                                 int hash_cap_in, int *coors_out, int *num_out_dev, int cap_out, int *nbr,
                                 unsigned long long *hash_keys_out, int *hash_vals_out, int hash_cap_out,
                                 void *workspace, size_t workspace_bytes, unsigned *row_mask, unsigned *status_dev,
                                 void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    ConvGeom g;
    // the input-side scatter enumerates at most ceil(k/s) <= 4 candidate outputs per dimension, which is only
    // right for dilation 1 (a dilated strided conv can reach more); SECOND never builds one (middle.py:146-189)
    B2S_REQUIRE(dilation == nullptr || (dilation[0] == 1 && dilation[1] == 1 && dilation[2] == 1) ||
                    (stride[0] == 1 && stride[1] == 1 && stride[2] == 1),
                "b2s_rulebook_conv: dilation > 1 combined with stride > 1 is not supported");
    B2S_REQUIRE(fill_geom(&g, in_shape, out_shape, ksize, stride, padding, dilation) == 0,
                "b2s_rulebook_conv: bad geometry");
    for (int j = 0; j < 3; ++j) {
        int expect = (g.in_shape[j] + 2 * g.p[j] - g.d[j] * (g.k[j] - 1) - 1) / g.s[j] + 1;
        B2S_REQUIRE(expect == g.out_shape[j], "b2s_rulebook_conv: out_shape[%d]=%d, expected %d", j,
                    g.out_shape[j], expect);
        B2S_REQUIRE((g.k[j] + g.s[j] - 1) / g.s[j] <= 4, "b2s_rulebook_conv: kernel/stride ratio > 4 in dim %d", j);
    }
    const bool want_hash = hash_keys_out != nullptr;      // NULL: the level's SubM table comes from b2s_rulebook_subm_ranked
    B2S_REQUIRE(!want_hash || ((hash_cap_out & (hash_cap_out - 1)) == 0 && hash_cap_out >= 2 * cap_out && hash_cap_out >= 2),
                "b2s_rulebook_conv: hash_cap_out must be a power of two >= 2*cap_out");
    ConvWorkspace w;
    size_t need = carve(&w, (char *)workspace, batch, out_shape);
    B2S_REQUIRE(workspace_bytes >= need, "b2s_rulebook_conv: workspace too small (%zu < %zu)", workspace_bytes, need);
    B2S_CUDA_OK(cudaMemsetAsync(w.bitmap, 0, sizeof(unsigned) * (size_t)(w.nwords + w.nsw), stream));
    if (row_mask && cap_out > 0) B2S_CUDA_OK(cudaMemsetAsync(row_mask, 0, sizeof(unsigned) * (size_t)cap_out, stream));
    if (want_hash) {
        B2S_CUDA_OK(cudaMemsetAsync(hash_keys_out, 0xFF, sizeof(unsigned long long) * (size_t)hash_cap_out, stream));
        B2S_CUDA_OK(cudaMemsetAsync(hash_vals_out, 0xFF, sizeof(int) * (size_t)hash_cap_out, stream));
    }
    if (cap_in > 0) {
        k_conv_mark<<<bounded_grid(cap_in, kThreads), kThreads, 0, stream>>>(coors_in, num_in_dev, cap_in, g, w.bitmap,
                                                                             w.summary);
        B2S_LAUNCH_OK();
    }
    // level 1: rank the non-empty words; level 2: rank the cells inside them
    k_summary_scan<<<w.nblk_s, kScanThreads, 0, stream>>>(w.summary, w.nsw, w.sum_prefix, w.sum_blocks);
    B2S_LAUNCH_OK();
    k_scan_sums<<<1, kScanThreads, 0, stream>>>(w.sum_blocks, w.nblk_s, nullptr, w.nnz, 0, nullptr);
    B2S_LAUNCH_OK();
    k_compact_words<<<bounded_grid(w.nsw, kThreads), kThreads, 0, stream>>>(w.summary, w.nsw, w.sum_prefix, w.sum_blocks,
                                                                            w.bitmap, w.nz_word, w.nz_prefix);
    B2S_LAUNCH_OK();
    k_nz_scan<<<bounded_grid(w.nwords, kScanThreads), kScanThreads, 0, stream>>>(w.nz_prefix, w.nnz, w.chunk_sums);
    B2S_LAUNCH_OK();
    k_scan_sums<<<1, kScanThreads, 0, stream>>>(w.chunk_sums, 0, w.nnz, num_out_dev, cap_out, status_dev);
    B2S_LAUNCH_OK();
    // B2S_RB_SCATTER=0: neighbour table by hash probes from the output side (k_conv_nbr), where an input hash exists.
    // The environment is read once; the choice is made per call, so a call without an input hash never changes it.
    static int env_scatter = -1;
    if (env_scatter < 0) { const char *e = getenv("B2S_RB_SCATTER"); env_scatter = (e && e[0] == '0') ? 0 : 1; }
    const int use_scatter = (env_scatter || !hash_keys_in) ? 1 : 0;
    k_conv_emit<<<bounded_grid(w.nwords < (1ll << 22) ? w.nwords : (1ll << 22), kThreads), kThreads, 0, stream>>>(
        w.bitmap, w.nz_word, w.nz_prefix, w.chunk_sums, w.nnz, g, cap_out, coors_out, use_scatter ? nbr : nullptr, w.wrow0);
    B2S_LAUNCH_OK();
    if (cap_out > 0) {
        if (want_hash) {
            k_hash_build<<<bounded_grid(cap_out, kThreads), kThreads, 0, stream>>>(
                coors_out, num_out_dev, cap_out, g.out_shape[0], g.out_shape[1], g.out_shape[2], hash_keys_out,
                hash_vals_out, hash_cap_out - 1, status_dev);
            B2S_LAUNCH_OK();
        }
        if (use_scatter && cap_in > 0) {
            k_conv_scatter_nbr<<<bounded_grid(cap_in, kThreads), kThreads, 0, stream>>>(
                coors_in, num_in_dev, cap_in, g, w.bitmap, w.wrow0, cap_out, nbr, row_mask);
        } else {
            k_conv_nbr<<<bounded_grid((long long)cap_out * g.K, kThreads), kThreads, 0, stream>>>(
                coors_out, num_out_dev, cap_out, g, hash_keys_in, hash_vals_in, hash_cap_in - 1, nbr, row_mask);
        }
        B2S_LAUNCH_OK();
    }
    return 0;
}

// SubM rulebook of the level b2s_rulebook_conv has JUST produced with this workspace (same batch and shape): the
// occupancy bitmap + per-word first rows are still there, so no hash table is needed for the level.
extern "C" int b2s_rulebook_subm_ranked(const int *coors, const int *num_rows_dev, int cap_rows, int batch,
                                        const int *shape, const int *ksize, const int *dilation, const void *workspace,
                                        size_t workspace_bytes, int *nbr, unsigned *row_mask, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    ConvGeom g;
    B2S_REQUIRE(fill_geom(&g, shape, nullptr, ksize, nullptr, nullptr, dilation) == 0,
                "b2s_rulebook_subm_ranked: bad geometry");
    B2S_REQUIRE((g.k[0] & 1) && (g.k[1] & 1) && (g.k[2] & 1), "b2s_rulebook_subm_ranked: kernel sizes must be odd");
    ConvWorkspace w;
    size_t need = carve(&w, (char *)workspace, batch, shape);
    B2S_REQUIRE(workspace_bytes >= need, "b2s_rulebook_subm_ranked: workspace too small (%zu < %zu)", workspace_bytes, need);
    if (cap_rows > 0) {
        B2S_CUDA_OK(cudaMemsetAsync(nbr, 0xFF, sizeof(int) * (size_t)cap_rows * g.K, stream));
        if (row_mask) B2S_CUDA_OK(cudaMemsetAsync(row_mask, 0, sizeof(unsigned) * (size_t)cap_rows, stream));
        k_subm_ranked<<<bounded_grid((long long)cap_rows * (g.K / 2 + 1), kThreads), kThreads, 0, stream>>>(
            coors, num_rows_dev, cap_rows, g, w.bitmap, w.wrow0, nbr, row_mask);
        B2S_LAUNCH_OK();
    }
    return 0;
}

extern "C" int b2s_rulebook_pairs(const int *nbr, const int *num_out_dev, int cap_out, int K, int L,
                                  int *indice_pairs, int *indice_pair_num, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (cap_out > 0 && K > 0) {
        k_pairs<<<bounded_grid((long long)cap_out * K, kThreads), kThreads, 0, stream>>>(nbr, num_out_dev, cap_out, K,
                                                                                     L, indice_pairs, indice_pair_num);
        B2S_LAUNCH_OK();
    }
    return 0;
}
