// csr.cu -- vertex-sorted view of a lattice set: for every lattice vertex the list of (point, barycentric
// weight) entries that splat onto it, IN POINT ORDER.
//
// The reference splats sequentially over points (permutohedral_cpu.h:653-661), so the float value of a
// vertex is the left-to-right sum of its contributions in point order.  Sorting the N*(d+1) entries by
// (vertex, point) once per lattice turns the splat into a segmented reduction over contiguous rows --
// no atomics, and a row walked front to back reproduces the reference's rounding bit for bit.
//
// Stable counting sort by vertex id, parallel over chunks of points:
//   k_csr_zero / k_csr_count   per-(chunk, vertex) entry counts                (integer atomics only)
//   k_csr_prefix               per vertex: exclusive prefix over its problem's chunks; row length
//   scan (3 launches)          row_ptr = exclusive scan of row lengths over all vertices of the batch
//   k_csr_fill                 every chunk walks its entries in scan order; warps commit in turn, lanes rank
//                              themselves with match.any, so equal vertices keep their point order
#include "engine.cuh"

namespace lccrf {

namespace {

constexpr int kFillThreads = 1024;
constexpr int kCursorSmemInts = 14336;  // 56 KB of shared cursors: lattices up to 14k vertices per problem

struct CsrParams {
    int G;                   // chunks
    int D;
    const int *chunk_prob;   // [G]
    const int *chunk_s0;     // [G] first entry (point*D) of the chunk
    const int *chunk_s1;     // [G] one past the last entry
    const long long *chunk_tbl;  // [G] base of the chunk's count row in tbl (stride = worst-case V of the problem)
    const int *prob_chunk0;  // [B+1] first chunk of each problem
    const int *offset;       // [NT*D] global vertex ids
    const float *bary;       // [NT*D]
    const int *vbase;        // [B+1]
    const int *vert_prob;    // [V]
    int *tbl;
    int *row_len;            // [Vcap+1] -> row_ptr after the scan
    int2 *ent;               // [NT*D] {point, bary bits} sorted by (vertex, point)
};

__global__ void __launch_bounds__(kThreads) k_csr_zero(CsrParams p) {
    const int g = blockIdx.x;
    const int b = __ldg(p.chunk_prob + g);
    const int Vb = __ldg(p.vbase + b + 1) - __ldg(p.vbase + b);
    int *row = p.tbl + __ldg(p.chunk_tbl + g);
    for (int v = threadIdx.x; v < Vb; v += kThreads) row[v] = 0;
}

__global__ void __launch_bounds__(kFillThreads) k_csr_count(CsrParams p) {
    const int g = blockIdx.x;
    const int b = __ldg(p.chunk_prob + g);
    const int vb = __ldg(p.vbase + b);
    int *row = p.tbl + __ldg(p.chunk_tbl + g);
    const int s0 = __ldg(p.chunk_s0 + g), s1 = __ldg(p.chunk_s1 + g);
    const unsigned lane = threadIdx.x & 31;
    for (int base = s0; base < s1; base += 4 * kFillThreads) {
        int v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int s = base + j * kFillThreads + threadIdx.x;
            v[j] = s < s1 ? __ldg(p.offset + s) - vb : -1;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const unsigned grp = __match_any_sync(0xffffffffu, v[j]);
            if (v[j] >= 0 && (__ffs(grp) - 1) == (int)lane) atomicAdd(row + v[j], __popc(grp));
        }
    }
}

__global__ void __launch_bounds__(kThreads) k_csr_prefix(CsrParams p, int B) {
    const int V = __ldg(p.vbase + B);
    for (int v = blockIdx.x * kThreads + threadIdx.x; v < V; v += gridDim.x * kThreads) {
        const int b = __ldg(p.vert_prob + v);
        const int lv = v - __ldg(p.vbase + b);
        const int g0 = __ldg(p.prob_chunk0 + b), g1 = __ldg(p.prob_chunk0 + b + 1);
        int run = 0;
        for (int g = g0; g < g1; g++) {
            int *c = p.tbl + __ldg(p.chunk_tbl + g) + lv;
            const int n = *c;
            *c = run;
            run += n;
        }
        p.row_len[v] = run;
    }
}

// ---- generic exclusive scan of ints whose length lives on the device (3 launches) ----
__global__ void __launch_bounds__(1024) k_scan_local(int *x, const int *n_ptr, int *blk_tot) {
    __shared__ int ws[32];
    const int n = __ldg(n_ptr);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int blk = blockIdx.x; blk * 1024 < n + 1; blk += gridDim.x) {  // n+1: the row_ptr sentinel
        const int idx = blk * 1024 + threadIdx.x;
        const int v = idx < n ? x[idx] : 0;
        int s = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane == 31) ws[wid] = s;
        __syncthreads();
        if (wid == 0) {
            int t = ws[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            ws[lane] = t;
        }
        __syncthreads();
        const int excl = (wid ? ws[wid - 1] : 0) + s - v;
        if (idx <= n) x[idx] = excl;
        if (threadIdx.x == 1023) blk_tot[blk] = ws[31];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_scan_tot(int *blk_tot, const int *n_ptr) {
    // exclusive scan of the block totals, single CTA (ceil((n+1)/1024) values)
    __shared__ int ws[32];
    __shared__ int carry_s;
    const int nblk = (__ldg(n_ptr) + 1 + 1023) / 1024;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int start = 0; start < nblk; start += 1024) {
        const int idx = start + threadIdx.x;
        const int v = idx < nblk ? blk_tot[idx] : 0;
        int s = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane == 31) ws[wid] = s;
        __syncthreads();
        if (wid == 0) {
            int t = ws[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            ws[lane] = t;
        }
        __syncthreads();
        const int carry = carry_s;
        if (idx < nblk) blk_tot[idx] = carry + (wid ? ws[wid - 1] : 0) + s - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + ws[31];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_scan_add(int *x, const int *n_ptr, const int *blk_tot) {
    const int n = __ldg(n_ptr);
    for (int blk = blockIdx.x; blk * 1024 < n + 1; blk += gridDim.x) {
        const int idx = blk * 1024 + threadIdx.x;
        if (idx <= n) x[idx] += __ldg(blk_tot + blk);
    }
}

// Stable placement.  A CTA owns one chunk; its kFillWarps warps own consecutive sub-chunks.
//   HIER (lattice of the problem has <= kHierV vertices): per-(warp, vertex) counts in shared memory, prefix over
//        the warps, then every warp walks its own sub-chunk in entry order with its own cursors -- no hand-offs.
//   otherwise: warp 0 walks the whole chunk in entry order with one cursor row (shared if it fits, else global).
// Inside a 32-entry group equal vertices are ranked by lane (= entry order) with match.any.
constexpr int kFillWarpsH = 8;
constexpr int kHierV = kCursorSmemInts / kFillWarpsH;  // 1792

constexpr int kFillAhead = 4;  // 32-entry groups whose loads are issued before the first one is consumed

template <int MODE>  // 0: hierarchical shared, 1: single warp + shared cursors, 2: single warp + global cursors
__device__ __forceinline__ void fill_walk(const CsrParams &p, int vb, int a, int z, int *cur_row, unsigned lane) {
    for (int base0 = a; base0 < z; base0 += 32 * kFillAhead) {
        // every load of kFillAhead groups is independent of the cursor logic: request them all, then commit in order
        int gv[kFillAhead], rp[kFillAhead];
        float w[kFillAhead];
#pragma unroll
        for (int g = 0; g < kFillAhead; g++) {
            const int s = base0 + 32 * g + (int)lane;
            gv[g] = s < z ? __ldg(p.offset + s) : -1;
            w[g] = s < z ? __ldg(p.bary + s) : 0.f;
        }
#pragma unroll
        for (int g = 0; g < kFillAhead; g++) rp[g] = gv[g] >= 0 ? __ldg(p.row_len + gv[g]) : 0;  // row_ptr after the scan
#pragma unroll
        for (int g = 0; g < kFillAhead; g++) {
            if (base0 + 32 * g >= z) break;  // (uniform)
            const int s = base0 + 32 * g + (int)lane;
            const int v = gv[g] >= 0 ? gv[g] - vb : -1;
            const unsigned grp = __match_any_sync(0xffffffffu, v);
            const int leader = __ffs(grp) - 1;
            const int rank = __popc(grp & ((1u << lane) - 1u));
            int cur = 0;
            if (v >= 0 && (int)lane == leader) {
                if (MODE == 2) {
                    cur = ((volatile int *)cur_row)[v];
                    ((volatile int *)cur_row)[v] = cur + __popc(grp);
                } else {
                    cur = cur_row[v];
                    cur_row[v] = cur + __popc(grp);
                }
            }
            __syncwarp();  // the next group may hit the same vertex
            cur = __shfl_sync(0xffffffffu, cur, leader);
            if (v >= 0) p.ent[rp[g] + cur + rank] = make_int2(s / p.D, __float_as_int(w[g]));
        }
    }
}

__global__ void __launch_bounds__(kFillWarpsH * 32) k_csr_fill(CsrParams p) {
    extern __shared__ int s_cur[];
    const int g = blockIdx.x;
    const int b = __ldg(p.chunk_prob + g);
    const int vb = __ldg(p.vbase + b);
    const int Vb = __ldg(p.vbase + b + 1) - vb;
    int *row = p.tbl + __ldg(p.chunk_tbl + g);
    const int s0 = __ldg(p.chunk_s0 + g), s1 = __ldg(p.chunk_s1 + g);
    const unsigned lane = threadIdx.x & 31;
    const int wid = threadIdx.x >> 5;
    if (Vb <= kHierV) {
        // sub-chunk of warp w: [s0 + w*sub, s0 + (w+1)*sub), sub a multiple of 32
        const int sub = ((s1 - s0 + kFillWarpsH - 1) / kFillWarpsH + 31) & ~31;
        const int a = min(s0 + wid * sub, s1), z = min(a + sub, s1);
        int *mine = s_cur + wid * Vb;
        for (int v = threadIdx.x; v < kFillWarpsH * Vb; v += kFillWarpsH * 32) s_cur[v] = 0;
        __syncthreads();
        for (int base0 = a; base0 < z; base0 += 32 * kFillAhead) {  // counts of this warp's sub-chunk
            int vv[kFillAhead];
#pragma unroll
            for (int g = 0; g < kFillAhead; g++) {
                const int s = base0 + 32 * g + (int)lane;
                vv[g] = s < z ? __ldg(p.offset + s) - vb : -1;
            }
#pragma unroll
            for (int g = 0; g < kFillAhead; g++) {
                const unsigned grp = __match_any_sync(0xffffffffu, vv[g]);
                if (vv[g] >= 0 && (__ffs(grp) - 1) == (int)lane) mine[vv[g]] += __popc(grp);
                __syncwarp();
            }
        }
        __syncthreads();
        for (int v = threadIdx.x; v < Vb; v += kFillWarpsH * 32) {  // exclusive prefix over the warps + chunk start
            int run = row[v];
#pragma unroll
            for (int w = 0; w < kFillWarpsH; w++) {
                const int n = s_cur[w * Vb + v];
                s_cur[w * Vb + v] = run;
                run += n;
            }
        }
        __syncthreads();
        fill_walk<0>(p, vb, a, z, mine, lane);
    } else if (wid == 0) {
        if (Vb <= kCursorSmemInts) {
            for (int v = (int)lane; v < Vb; v += 32) s_cur[v] = row[v];
            __syncwarp();
            fill_walk<1>(p, vb, s0, s1, s_cur, lane);
        } else {
            fill_walk<2>(p, vb, s0, s1, row, lane);
        }
    }
}

// rows by length class: long rows (>= kLongRow entries) go to the speculative scan; the short ones are grouped
// into pieces (a diagnostic of the row structure since k_splat_rows works by fixed entry tiles) -- a piece starts at a
// short row that is the first row, follows a long row, or is the first to start in its granule of kTileGranule
// entries.  List order is irrelevant: rows / pieces are independent.
__global__ void __launch_bounds__(kThreads)
k_row_classify(const int *__restrict__ row_ptr, const int *__restrict__ vtotal, int *__restrict__ lng,
               int *__restrict__ counts, int *__restrict__ piece_list) {
    const int V = __ldg(vtotal);
    for (int v = blockIdx.x * kThreads + threadIdx.x; v < V; v += gridDim.x * kThreads) {
        const int start = __ldg(row_ptr + v);
        const int len = __ldg(row_ptr + v + 1) - start;
        if (len >= kLongRow) {
            lng[atomicAdd(counts, 1)] = v;
        } else {
            bool first = v == 0;
            if (!first) {
                const int pstart = __ldg(row_ptr + v - 1);
                first = (start - pstart >= kLongRow) || (start / kTileGranule != pstart / kTileGranule);
            }
            if (first) piece_list[atomicAdd(counts + 2, 1)] = v;
        }
    }
}

// chunks of the long rows: long_chunk0 = exclusive scan of ceil(len / kScanChunk) over the long list, chunk_row[c] =
// list index of the row that owns chunk c, counts[1] = number of chunks.  Single CTA (the list is short).
__global__ void __launch_bounds__(1024)
k_long_chunks(const int *__restrict__ row_ptr, const int *__restrict__ lng, int *__restrict__ counts,
              int *__restrict__ long_chunk0, int4 *__restrict__ chunk_desc) {
    __shared__ int ws[32];
    __shared__ int carry_s;
    const int n = counts[0];
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int start = 0; start < n; start += 1024) {
        const int i = start + threadIdx.x;
        int nch = 0, rs = 0, re = 0;
        if (i < n) {
            const int v = lng[i];
            rs = __ldg(row_ptr + v);
            re = __ldg(row_ptr + v + 1);
            nch = (re - rs + kScanChunk - 1) / kScanChunk;
        }
        int x = nch;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) ws[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int t = ws[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            ws[lane] = t;
        }
        __syncthreads();
        const int carry = carry_s;
        const int base = carry + (wid ? ws[wid - 1] : 0) + x - nch;
        if (i < n) {
            long_chunk0[i] = base;
            for (int c = 0; c < nch; c++)
                chunk_desc[base + c] = make_int4(rs + c * kScanChunk, min(rs + (c + 1) * kScanChunk, re), base, i);
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + ws[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        long_chunk0[n] = carry_s;
        counts[1] = carry_s;
    }
}

// tile_row0[t] = the (non-empty) row that holds entry t * kTreeTile; tile_row0[n_tiles] = V - 1 (k_splat_tree, k_splat_rows);
// tile_own[t] != 0 iff the ordered short-row splat has work in tile t: a row shorter than kLongRow starts there, or a row
// without entries belongs to it (same ownership rule as k_splat_rows)
__global__ void __launch_bounds__(kThreads)
k_tile_rows(const int *__restrict__ row_ptr, const int *__restrict__ vtotal, int *__restrict__ tile_row0,
            int *__restrict__ tile_own, int n_tiles) {
    const int V = __ldg(vtotal);
    if (blockIdx.x == 0 && threadIdx.x == 0) tile_row0[n_tiles] = V - 1;
    for (int v = blockIdx.x * kThreads + threadIdx.x; v < V; v += gridDim.x * kThreads) {
        const int s = __ldg(row_ptr + v), e = __ldg(row_ptr + v + 1);
        for (int t = (s + kTreeTile - 1) / kTreeTile; t < n_tiles && t * kTreeTile < e; t++) tile_row0[t] = v;
        if (e - s < kLongRow && n_tiles > 0) {
            const int t = e > s ? s / kTreeTile : (s > 0 ? (s - 1) / kTreeTile : 0);
            tile_own[t < n_tiles ? t : n_tiles - 1] = 1;
        }
    }
}

}  // namespace

int csr_create(Ctx *ctx, const Batch &b, LatticeSet *ls) {
    const int D = ls->D;
    std::vector<int> chunk_prob, chunk_s0, chunk_s1, prob_chunk0(b.B + 1);
    std::vector<long long> chunk_tbl;
    long long tbl = 0;
    // The chunk size sets the parallelism of the sort, not its result (rows keep point order either way).  A batch of
    // many image-sized problems whose tables together exceed 2^31 entries takes coarser chunks in every problem.
    for (long long min_cpts = kCsrChunkPoints;; min_cpts *= 2) {
        chunk_prob.clear();
        chunk_s0.clear();
        chunk_s1.clear();
        chunk_tbl.clear();
        tbl = 0;
        for (int i = 0; i < b.B; i++) {
            prob_chunk0[i] = (int)chunk_prob.size();
            const int p0 = b.h_prob_ptr[i], p1 = b.h_prob_ptr[i + 1];
            const long long stride = ((long long)(p1 - p0) + 1) * D;  // worst-case vertex count of the problem
            // the count table is chunks x vertices: image-scale problems (millions of points) take coarser chunks so
            // that one problem's table stays below 2^30 entries
            long long cpts = min_cpts;
            while (((long long)(p1 - p0) + cpts - 1) / cpts * stride > (1ll << 30)) cpts *= 2;
            for (long long c = p0; c < p1; c += cpts) {
                chunk_prob.push_back(i);
                chunk_s0.push_back((int)(c * D));
                chunk_s1.push_back((int)((c + cpts < p1 ? c + cpts : p1) * D));
                chunk_tbl.push_back(tbl);
                tbl += stride;
            }
        }
        if (tbl <= (1ll << 31) - 1 || min_cpts > b.maxN) break;
    }
    prob_chunk0[b.B] = (int)chunk_prob.size();
    ls->csr_chunks = (int)chunk_prob.size();
    if (tbl > (1ll << 31) - 1) return fail(LCCRF_ERR_ARG, "CSR count table would exceed 2^31 entries");
    const size_t G = (size_t)(ls->csr_chunks > 0 ? ls->csr_chunks : 1);
    int rc = LCCRF_OK;
    rc |= dev_alloc(ctx, (void **)&ls->chunk_prob, G * 4);
    rc |= dev_alloc(ctx, (void **)&ls->chunk_s0, G * 4);
    rc |= dev_alloc(ctx, (void **)&ls->chunk_s1, G * 4);
    rc |= dev_alloc(ctx, (void **)&ls->chunk_tbl, G * 8);
    rc |= dev_alloc(ctx, (void **)&ls->prob_chunk0, (size_t)(b.B + 1) * 4);
    rc |= dev_alloc(ctx, (void **)&ls->csr_tbl, (size_t)(tbl > 0 ? tbl : 1) * 4);
    rc |= dev_alloc(ctx, (void **)&ls->row_ptr, ((size_t)ls->Vcap + 2) * 4);
    rc |= dev_alloc(ctx, (void **)&ls->csr_ent, (size_t)(b.NT > 0 ? b.NT : 1) * D * sizeof(int2));
    rc |= dev_alloc(ctx, (void **)&ls->scan_tot, ((size_t)ls->Vcap / 1024 + 2) * 4);
    {   // long rows: at most E / kLongRow of them; their chunks: at most E / kScanChunk full ones + one partial per row
        const long long E = (long long)b.NT * D;
        ls->max_long = (int)(E / kLongRow);
        ls->max_chunks = (int)(E / kScanChunk) + ls->max_long;
    }
    rc |= dev_alloc(ctx, (void **)&ls->row_list_long, ((size_t)ls->max_long + 1) * 4);
    rc |= dev_alloc(ctx, (void **)&ls->long_chunk0, ((size_t)ls->max_long + 2) * 4);
    rc |= dev_alloc(ctx, (void **)&ls->chunk_desc, ((size_t)ls->max_chunks + 1) * 16);
    rc |= dev_alloc(ctx, (void **)&ls->row_counts, 16 * 4, true);  // [8..15] live across lattice builds (filter.cu)
    ls->max_pieces = (int)(((long long)b.NT * D) / kTileGranule + ((long long)b.NT * D) / kLongRow + 2);
    rc |= dev_alloc(ctx, (void **)&ls->piece_list, (size_t)ls->max_pieces * 4);
    ls->n_tiles = (int)(((long long)b.NT * D + kTreeTile - 1) / kTreeTile);
    rc |= dev_alloc(ctx, (void **)&ls->tile_row0, ((size_t)ls->n_tiles + 1) * 4);
    rc |= dev_alloc(ctx, (void **)&ls->tile_own, ((size_t)ls->n_tiles + 1) * 4);
    rc |= dev_alloc(ctx, (void **)&ls->tile_info, ((size_t)ls->n_tiles + 1) * sizeof(int2));
    if (ls->Lmax > 0) rc |= dev_alloc(ctx, (void **)&ls->tile_part, ((size_t)ls->n_tiles + 1) * ls->Lmax * sizeof(float));
    if (rc != LCCRF_OK) return LCCRF_ERR_CUDA;
    cudaStream_t st = ctx->stream;
    if (ls->csr_chunks > 0) {
        LCCRF_CUDA(cudaMemcpyAsync(ls->chunk_prob, chunk_prob.data(), G * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(ls->chunk_s0, chunk_s0.data(), G * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(ls->chunk_s1, chunk_s1.data(), G * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(ls->chunk_tbl, chunk_tbl.data(), G * 8, cudaMemcpyHostToDevice, st));
    }
    LCCRF_CUDA(cudaMemcpyAsync(ls->prob_chunk0, prob_chunk0.data(), (size_t)(b.B + 1) * 4, cudaMemcpyHostToDevice, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));  // host vectors go out of scope
    return LCCRF_OK;
}

void csr_destroy(Ctx *ctx, LatticeSet *ls) {
    dev_free(ctx, ls->chunk_prob);
    dev_free(ctx, ls->chunk_s0);
    dev_free(ctx, ls->chunk_s1);
    dev_free(ctx, ls->chunk_tbl);
    dev_free(ctx, ls->prob_chunk0);
    dev_free(ctx, ls->csr_tbl);
    dev_free(ctx, ls->row_ptr);
    dev_free(ctx, ls->csr_ent);
    dev_free(ctx, ls->scan_tot);
    dev_free(ctx, ls->row_list_long);
    dev_free(ctx, ls->long_chunk0);
    dev_free(ctx, ls->chunk_desc);
    dev_free(ctx, ls->chunk_sum);
    dev_free(ctx, ls->chunk_rec);
    dev_free(ctx, ls->row_counts);
    dev_free(ctx, ls->piece_list);
    dev_free(ctx, ls->tile_row0);
    dev_free(ctx, ls->tile_own);
    dev_free(ctx, ls->tile_info);
    dev_free(ctx, ls->tile_part);
}

int csr_build(Ctx *ctx, const Batch &b, LatticeSet *ls) {
    cudaStream_t st = ctx->stream;
    CsrParams p;
    p.G = ls->csr_chunks;
    p.D = ls->D;
    p.chunk_prob = ls->chunk_prob;
    p.chunk_s0 = ls->chunk_s0;
    p.chunk_s1 = ls->chunk_s1;
    p.chunk_tbl = ls->chunk_tbl;
    p.prob_chunk0 = ls->prob_chunk0;
    p.offset = ls->offset;
    p.bary = ls->bary;
    p.vbase = ls->vbase;
    p.vert_prob = ls->vert_prob;
    p.tbl = ls->csr_tbl;
    p.row_len = ls->row_ptr;
    p.ent = ls->csr_ent;
    const int *vt = ls->vbase + ls->B;
    if (p.G > 0) {
        { LCCRF_KERNEL(ctx, "k_csr_zero"); k_csr_zero<<<p.G, kThreads, 0, st>>>(p); }
        { LCCRF_KERNEL(ctx, "k_csr_count"); k_csr_count<<<p.G, kFillThreads, 0, st>>>(p); }
    }
    const int vgrid = persistent_grid((long long)ls->Vcap, kThreads, 4);
    { LCCRF_KERNEL(ctx, "k_csr_prefix"); k_csr_prefix<<<vgrid, kThreads, 0, st>>>(p, b.B); }
    const int sgrid = persistent_grid((long long)ls->Vcap + 1, 1024, 2);
    { LCCRF_KERNEL(ctx, "k_scan_local"); k_scan_local<<<sgrid, 1024, 0, st>>>(ls->row_ptr, vt, ls->scan_tot); }
    { LCCRF_KERNEL(ctx, "k_scan_tot"); k_scan_tot<<<1, 1024, 0, st>>>(ls->scan_tot, vt); }
    { LCCRF_KERNEL(ctx, "k_scan_add"); k_scan_add<<<sgrid, 1024, 0, st>>>(ls->row_ptr, vt, ls->scan_tot); }
    if (p.G > 0) {
        LCCRF_TRY(ensure_dyn_smem(ctx, k_csr_fill, kCursorSmemInts * (int)sizeof(int)));
        { LCCRF_KERNEL(ctx, "k_csr_fill"); k_csr_fill<<<p.G, kFillWarpsH * 32, kCursorSmemInts * sizeof(int), st>>>(p); }
    }
    LCCRF_CUDA(cudaMemsetAsync(ls->row_counts, 0, 8 * sizeof(int), st));
    { LCCRF_KERNEL(ctx, "k_row_classify"); k_row_classify<<<vgrid, kThreads, 0, st>>>(ls->row_ptr, vt, ls->row_list_long, ls->row_counts, ls->piece_list); }
    if (ls->max_long > 0) {
        LCCRF_KERNEL(ctx, "k_long_chunks");
        k_long_chunks<<<1, 1024, 0, st>>>(ls->row_ptr, ls->row_list_long, ls->row_counts, ls->long_chunk0, (int4 *)ls->chunk_desc);
    }
    if (ls->n_tiles > 0) {
        LCCRF_CUDA(cudaMemsetAsync(ls->tile_own, 0, (size_t)ls->n_tiles * sizeof(int), st));
        LCCRF_KERNEL(ctx, "k_tile_rows");
        k_tile_rows<<<vgrid, kThreads, 0, st>>>(ls->row_ptr, vt, ls->tile_row0, ls->tile_own, ls->n_tiles);
    }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

}  // namespace lccrf
