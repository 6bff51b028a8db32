// lattice_build.cu -- permutohedral lattice construction on the GPU, bit-exact with
// PermutohedralLatticeCPU::init (Thirdparty/DenseCRF/include/permutohedral_cpu.h:241-424, SSE branch).
//
//   k_embed<d>    elevate / round / rank / barycentric / keys for every point (incl. the reference's
//                 phantom lanes, :294-299) and atomicCAS insertion of each key into a per-problem
//                 open-addressing region; atomicMin records the FIRST scan position of every vertex.
//   k_vertex_ids  canonical ids: the reference's id of a vertex is the number of distinct keys whose
//                 first occurrence precedes its own in the k-major / remainder-minor scan (:371-377,
//                 HashTableCPU::find :146).  That is an exclusive prefix sum over "is first occurrence"
//                 flags in scan order -- no sort needed, and ids are bit-identical to the reference.
//                 One launch: a chained scan with decoupled look-back.
//   k_offsets     offset_[point][remainder] = id
//   k_neighbours<d>  blur_neighbors_ (:408-421) by hash lookups of key -/+ 1 (axis j: +/- d)
//   k_hash_clear<d>  empties the slots the build used, so the hash regions need no clear before the next build
//
// All arithmetic of the embedding is IEEE fp32 with every operation individually rounded
// (__fmul_rn/__fadd_rn/__fsub_rn, file compiled with -fmad=false): the reference is built without
// FMA (CMakeLists.txt:11-12) and rounds half-to-even (cvtps_epi32 under MXCSR nearest, :289-290,319).
#include <climits>
#include <cmath>
#include <cstring>

#include "engine.cuh"

namespace lccrf {

namespace {

constexpr uint64_t kTag = 1ull << 63;  // every stored key word has bit 63 set, so 0 == empty

__host__ __device__ constexpr int num_levels(int d) { return d <= 3 ? 1 : 1 + (d - 3 + 1) / 2; }

struct BuildParams {
    int NT, B;
    const int *prob_ptr;   // [B+1]
    const int *tab_base;   // [B+1] first slot of each problem's hash region (sizes are powers of two)
    const float *feat;     // [NT*d]
    uint64_t *key[3];      // key words per level
    int *first;            // [slots] first scan position of the vertex stored in a last-level slot
    int *tab_id;           // [slots] global vertex id of a last-level slot
    int *ent_slot;         // [(NT+B)*D] last-level slot per scan position, -1 for inactive phantom entries
    float *bary;           // [NT*D]
    int *offset;           // [NT*D]
    int2 *nbr;             // [D][Vcap]
    int *vert_slot, *vert_prob, *vbase;
    int Vcap;
    int *status;
    float scale[LCCRF_MAX_D];
    float invD, fD;
};

__device__ __forceinline__ int hash_insert(uint64_t *keys, int base, uint32_t mask, uint64_t word) {
    uint32_t h = mix64(word) & mask;
    for (;;) {
        uint64_t prev = __ldcg((const unsigned long long *)keys + base + h);
        if (prev == word) return base + (int)h;
        if (prev == 0ull) {
            prev = atomicCAS((unsigned long long *)keys + base + h, 0ull, (unsigned long long)word);
            if (prev == 0ull || prev == word) return base + (int)h;
        }
        h = (h + 1) & mask;
    }
}

__device__ __forceinline__ int hash_find(const uint64_t *keys, int base, uint32_t mask, uint64_t word) {
    uint32_t h = mix64(word) & mask;
    for (;;) {
        uint64_t k = __ldg((const unsigned long long *)keys + base + h);
        if (k == word) return base + (int)h;
        if (k == 0ull) return -1;
        h = (h + 1) & mask;
    }
}

// key words: level 0 packs coords 0..2, each further level packs the previous level's region-local
// slot (31 bits) with two more coords.  d <= 3: one level; d in {4,5}: two; d in {6,7}: three.
template <int d>
__device__ __forceinline__ uint64_t word_level(const int *kc, int lev, int prev_local_slot) {
    if (lev == 0) {
        uint64_t w = kTag | (uint64_t)(uint16_t)kc[0];
        if (d > 1) w |= (uint64_t)(uint16_t)kc[1] << 16;
        if (d > 2) w |= (uint64_t)(uint16_t)kc[2] << 32;
        return w;
    }
    int c0 = 3 + 2 * (lev - 1);
    uint64_t w = kTag | ((uint64_t)(uint32_t)prev_local_slot << 32) | (uint64_t)(uint16_t)kc[c0];
    if (c0 + 1 < d) w |= (uint64_t)(uint16_t)kc[c0 + 1] << 16;
    return w;
}

__device__ __forceinline__ int pseudo_problem(const int *__restrict__ prob_ptr, int B, int ip) {
    int lo = 0, hi = B;  // pp[b] = prob_ptr[b] + b, strictly increasing
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (__ldg(prob_ptr + mid) + mid <= ip) lo = mid;
        else hi = mid;
    }
    return lo;
}

template <int d>
__global__ void __launch_bounds__(kThreads) k_embed(BuildParams p) {
    constexpr int D = d + 1;
    constexpr int NLEV = num_levels(d);
    const int ip = blockIdx.x * kThreads + threadIdx.x;  // pseudo-point index in scan space
    if (ip >= p.NT + p.B) return;
    const int b = pseudo_problem(p.prob_ptr, p.B, ip);
    const int p0 = __ldg(p.prob_ptr + b), p1 = __ldg(p.prob_ptr + b + 1);
    const int Nb = p1 - p0;
    const int local = ip - (p0 + b);
    const bool phantom = (local == Nb);
    int *es = p.ent_slot + (size_t)ip * D;
    if (phantom && (Nb & 3) == 0) {  // no padding lanes in the reference's last block of four
#pragma unroll
        for (int r = 0; r < D; r++) es[r] = -1;
        return;
    }
    const int i = p0 + local;
    float f[d];
#pragma unroll
    for (int j = 0; j < d; j++) f[j] = phantom ? 0.0f : __ldg(p.feat + (size_t)i * d + j);

    // elevate (:304-310)
    float el[D];
    float sm = 0.0f;
#pragma unroll
    for (int j = d; j > 0; j--) {
        float cf = __fmul_rn(f[j - 1], p.scale[j - 1]);
        el[j] = __fsub_rn(sm, __fmul_rn((float)j, cf));
        sm = __fadd_rn(sm, cf);
    }
    el[0] = sm;
    // nearest 0-coloured simplex (:313-323), round half to even
    float rem[D];
    int rank[D];
    int sum = 0;
#pragma unroll
    for (int q = 0; q < D; q++) {
        float v = rintf(__fmul_rn(p.invD, el[q]));
        rem[q] = __fmul_rn(v, p.fD);
        sum += (int)v;
        rank[q] = 0;
    }
    // rank (:326-336), ties to the higher index
#pragma unroll
    for (int a = 0; a < d; a++) {
        float da = __fsub_rn(el[a], rem[a]);
#pragma unroll
        for (int c = a + 1; c < D; c++) {
            float dc = __fsub_rn(el[c], rem[c]);
            if (da < dc) rank[a]++;
            else rank[c]++;
        }
    }
    // back onto the plane (:339-345)
#pragma unroll
    for (int q = 0; q < D; q++) {
        rank[q] += sum;
        if (rank[q] < 0) {
            rank[q] += D;
            rem[q] = __fadd_rn(rem[q], p.fD);
        } else if (rank[q] >= D) {
            rank[q] -= D;
            rem[q] = __fsub_rn(rem[q], p.fD);
        }
    }
    // barycentric (:348-366), literal update order (i ascending, += then -=) via predicated selects
    float bc[D + 1];
#pragma unroll
    for (int q = 0; q <= D; q++) bc[q] = 0.0f;
#pragma unroll
    for (int a = 0; a < D; a++) {
        float v = __fmul_rn(__fsub_rn(el[a], rem[a]), p.invD);
        int pi = d - rank[a];
#pragma unroll
        for (int q = 0; q <= D; q++) {
            if (q == pi) bc[q] = __fadd_rn(bc[q], v);
            if (q == pi + 1) bc[q] = __fsub_rn(bc[q], v);
        }
    }
    bc[0] = __fadd_rn(bc[0], __fadd_rn(1.0f, bc[D]));

    // keys + insertion (:371-377)
    const int base = __ldg(p.tab_base + b);
    const uint32_t mask = (uint32_t)(__ldg(p.tab_base + b + 1) - base) - 1u;
    bool range_ok = true;
#pragma unroll
    for (int r = 0; r < D; r++) {
        int kc[d];
#pragma unroll
        for (int c = 0; c < d; c++) {
            kc[c] = (int)rem[c] + ((rank[c] <= d - r) ? r : r - D);
            range_ok = range_ok && (kc[c] >= -32768 && kc[c] <= 32767);
        }
        int slot = 0;
#pragma unroll
        for (int lev = 0; lev < NLEV; lev++) {
            uint64_t w = word_level<d>(kc, lev, slot - base);
            slot = hash_insert(p.key[lev], base, mask, w);
        }
        // most points find an earlier first occurrence already recorded: skip the atomic (hot vertices
        // would otherwise serialise tens of thousands of atomicMin on one address)
        if (__ldcg(p.first + slot) > ip * D + r) atomicMin(p.first + slot, ip * D + r);
        es[r] = slot;
        if (!phantom) p.bary[(size_t)i * D + r] = bc[r];
    }
    if (!range_ok) atomicOr(p.status, 1);
}

// ---- canonical ids: exclusive scan of "first occurrence" flags over scan positions ----
__device__ __forceinline__ bool is_first(const BuildParams &p, int s, int S, int &slot) {
    slot = -1;
    if (s >= S) return false;
    slot = __ldg(p.ent_slot + s);
    return slot >= 0 && __ldg(p.first + slot) == s;
}

// Single-pass chained scan (decoupled look-back).  A tile of kIdTile scan positions counts its flags, publishes the
// count, adds the counts / prefixes of the tiles in front and publishes its inclusive prefix.  Tiles are numbered by an
// atomic ticket, so a tile only ever waits on tiles that are already running.  The status words and the ticket
// (ids_status, cleared before every launch) hold {flag (1: count, 2: inclusive prefix), value}.
constexpr int kIdThreads = 1024;
constexpr int kIdItems = 4;
constexpr int kIdTile = kIdThreads * kIdItems;
constexpr unsigned long long kIdCount = 1ull << 32, kIdPrefix = 2ull << 32;

__device__ __forceinline__ void id_publish(unsigned long long *p, unsigned long long w) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
__device__ __forceinline__ unsigned long long id_poll(const unsigned long long *p) {
    unsigned long long w;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
    return w;
}

// writes tab_id, vert_slot, vert_prob, vbase[0..B]
template <int D>
__global__ void __launch_bounds__(kIdThreads) k_vertex_ids(BuildParams p, unsigned long long *ids_status, int ntiles) {
    __shared__ int s_excl[kIdItems * 32];       // per 32-position group (scan order): flags in front of it inside the tile
    __shared__ unsigned s_bal[kIdItems * 32];   // per group: its flags
    __shared__ int s_tile, s_prefix, s_total;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ids_status + ntiles, 1ull);
    __syncthreads();
    const int tile = s_tile;
    const int S = (p.NT + p.B) * D;
    const int s0 = tile * kIdTile;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int slot[kIdItems];
    unsigned bal[kIdItems];
#pragma unroll
    for (int j = 0; j < kIdItems; j++) {
        const bool f = is_first(p, s0 + j * kIdThreads + threadIdx.x, S, slot[j]);
        bal[j] = __ballot_sync(0xffffffffu, f);
        if (!f) slot[j] = -1;
        if (lane == 0) s_bal[j * 32 + wid] = bal[j];
    }
    __syncthreads();
    if (wid == 0) {
        int c[kIdItems], sum = 0;
#pragma unroll
        for (int k = 0; k < kIdItems; k++) {
            c[k] = __popc(s_bal[lane * kIdItems + k]);
            sum += c[k];
        }
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        int run = incl - sum;
#pragma unroll
        for (int k = 0; k < kIdItems; k++) {
            s_excl[lane * kIdItems + k] = run;
            run += c[k];
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        int prefix = 0;
        if (tile > 0) {
            if (lane == 0) id_publish(ids_status + tile, kIdCount | (unsigned)total);
            for (int pred = tile - 1;;) {
                const int t = pred - lane;
                const unsigned long long w = t >= 0 ? id_poll(ids_status + t) : kIdPrefix;
                if (__any_sync(0xffffffffu, (w >> 32) == 0)) continue;  // a tile in the window has not published yet
                const unsigned pm = __ballot_sync(0xffffffffu, (w >> 32) == 2);
                const int stop = pm ? __ffs(pm) - 1 : 31;  // nearest inclusive prefix ends the walk
                int v = lane <= stop ? (int)(unsigned)w : 0;
#pragma unroll
                for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                prefix += v;
                if (pm) break;
                pred -= 32;
            }
        }
        if (lane == 0) {
            id_publish(ids_status + tile, kIdPrefix | (unsigned)(prefix + total));
            s_prefix = prefix;
            s_total = total;
        }
    }
    __syncthreads();
    const int prefix = s_prefix;
#pragma unroll
    for (int j = 0; j < kIdItems; j++) {
        if (slot[j] >= 0) {
            const int s = s0 + j * kIdThreads + threadIdx.x;
            const int id = prefix + s_excl[j * 32 + wid] + __popc(bal[j] & ((1u << lane) - 1u));
            p.tab_id[slot[j]] = id;
            p.vert_slot[id] = slot[j];
            p.vert_prob[id] = pseudo_problem(p.prob_ptr, p.B, s / D);
        }
    }
    // vbase[b] = number of first occurrences in front of problem b's first scan position (the phantom point keeps
    // every problem's first position inside [0, S), so exactly one tile writes it)
    const int s1 = s0 + kIdTile;
    const int b0 = s0 < S ? pseudo_problem(p.prob_ptr, p.B, s0 / D) : p.B;
    for (int b = b0 + (int)threadIdx.x; b < p.B; b += kIdThreads) {
        const int sb = (__ldg(p.prob_ptr + b) + b) * D;
        if (sb >= s1) break;
        if (sb >= s0) {
            const int q = sb - s0, g = q >> 5;
            p.vbase[b] = prefix + s_excl[g] + __popc(s_bal[g] & ((1u << (q & 31)) - 1u));
        }
    }
    if (tile == ntiles - 1 && threadIdx.x == 0) p.vbase[p.B] = prefix + s_total;
}

template <int D>
__global__ void __launch_bounds__(kThreads) k_offsets(BuildParams p) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= p.NT) return;
    const int b = find_segment(p.prob_ptr, p.B + 1, i);
    const int *es = p.ent_slot + (size_t)(i + b) * D;
#pragma unroll
    for (int r = 0; r < D; r++) p.offset[(size_t)i * D + r] = __ldg(p.tab_id + __ldg(es + r));
}

template <int d>
__global__ void __launch_bounds__(kThreads) k_neighbours(BuildParams p) {
    constexpr int D = d + 1;
    constexpr int NLEV = num_levels(d);
    const int V = __ldg(p.vbase + p.B);
    const long long total = (long long)V * D;
    for (long long t = (long long)blockIdx.x * kThreads + threadIdx.x; t < total;
         t += (long long)gridDim.x * kThreads) {
        const int j = (int)(t / V), id = (int)(t - (long long)j * V);
        const int b = __ldg(p.vert_prob + id);
        const int base = __ldg(p.tab_base + b);
        const uint32_t mask = (uint32_t)(__ldg(p.tab_base + b + 1) - base) - 1u;
        // reconstruct the key by walking the level chain backwards
        int kc[d];
        int slot = __ldg(p.vert_slot + id);
#pragma unroll
        for (int lev = NLEV - 1; lev >= 0; lev--) {
            uint64_t w = __ldg((const unsigned long long *)p.key[lev] + slot);
            if (lev == 0) {
                kc[0] = (short)(w & 0xffff);
                if (d > 1) kc[1] = (short)((w >> 16) & 0xffff);
                if (d > 2) kc[2] = (short)((w >> 32) & 0xffff);
            } else {
                int c0 = 3 + 2 * (lev - 1);
                kc[c0] = (short)(w & 0xffff);
                if (c0 + 1 < d) kc[c0 + 1] = (short)((w >> 16) & 0xffff);
                slot = base + (int)((w >> 32) & 0x7fffffffu);
            }
        }
        int res[2];
#pragma unroll
        for (int side = 0; side < 2; side++) {
            int nk[d];
#pragma unroll
            for (int c = 0; c < d; c++) {
                int v = side == 0 ? kc[c] - 1 : kc[c] + 1;              // :412-413
                if (c == j) v = side == 0 ? kc[c] + d : kc[c] - d;      // :415-416 (j == d touches no hashed coord)
                nk[c] = (int)(short)v;                                   // short arithmetic wraps
            }
            int sl = base;
            bool found = true;
#pragma unroll
            for (int lev = 0; lev < NLEV; lev++) {
                if (found) {
                    uint64_t w = word_level<d>(nk, lev, sl - base);
                    sl = hash_find(p.key[lev], base, mask, w);
                    found = sl >= 0;
                }
            }
            res[side] = found ? __ldg(p.tab_id + sl) : -1;
        }
        p.nbr[(size_t)j * p.Vcap + id] = make_int2(res[0], res[1]);
    }
}

// Return the slots this build used to the empty state (key 0, first 0x7f7f7f7f): the last-level slot of every vertex
// and, for d >= 4, the slots of its key chain at the earlier levels.  Those are shared between vertices; atomicExch
// lets exactly one of the threads that reach a slot read its link to the level below.
template <int d>
__global__ void __launch_bounds__(kThreads) k_hash_clear(BuildParams p) {
    constexpr int NLEV = num_levels(d);
    const int V = __ldg(p.vbase + p.B);
    for (int id = blockIdx.x * kThreads + threadIdx.x; id < V; id += gridDim.x * kThreads) {
        int slot = __ldg(p.vert_slot + id);
        p.first[slot] = 0x7f7f7f7f;
        if (NLEV == 1) {
            p.key[0][slot] = 0ull;
            continue;
        }
        const int base = __ldg(p.tab_base + __ldg(p.vert_prob + id));
        uint64_t w = p.key[NLEV - 1][slot];
        p.key[NLEV - 1][slot] = 0ull;
#pragma unroll
        for (int lev = NLEV - 2; lev >= 0 && w != 0ull; lev--) {
            slot = base + (int)((w >> 32) & 0x7fffffffu);
            w = atomicExch((unsigned long long *)p.key[lev] + slot, 0ull);
        }
    }
}

template <int d>
int launch_build(Ctx *ctx, const BuildParams &p, unsigned long long *ids_status) {
    constexpr int D = d + 1;
    cudaStream_t st = ctx->stream;
    const int NP = p.NT + p.B;
    const long long S = (long long)NP * D;
    const int ntiles = S > 0 ? cdiv(S, kIdTile) : 1;
    const int vgrid = persistent_grid((long long)p.Vcap, kThreads, 4);
    { LCCRF_KERNEL(ctx, "k_embed"); k_embed<d><<<cdiv(NP, kThreads), kThreads, 0, st>>>(p); }
    LCCRF_CUDA(cudaMemsetAsync(ids_status, 0, ((size_t)ntiles + 1) * sizeof(unsigned long long), st));
    { LCCRF_KERNEL(ctx, "k_vertex_ids"); k_vertex_ids<D><<<ntiles, kIdThreads, 0, st>>>(p, ids_status, ntiles); }
    if (p.NT > 0) {
        { LCCRF_KERNEL(ctx, "k_offsets"); k_offsets<D><<<cdiv(p.NT, kThreads), kThreads, 0, st>>>(p); }
    }
    { LCCRF_KERNEL(ctx, "k_neighbours"); k_neighbours<d><<<vgrid, kThreads, 0, st>>>(p); }
    { LCCRF_KERNEL(ctx, "k_hash_clear"); k_hash_clear<d><<<vgrid, kThreads, 0, st>>>(p); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

}  // namespace

int lattice_set_create(Ctx *ctx, const Batch &b, int d, float w, int Lmax, LatticeSet **out) {
    if (d < 1 || d > LCCRF_MAX_D) return fail(LCCRF_ERR_ARG, "feature dimension must be in [1, LCCRF_MAX_D]");
    auto *ls = new LatticeSet();
    ls->d = d;
    ls->D = d + 1;
    ls->w = w;
    ls->alpha = 1.0f / (1 + powf(2, (float)-d));  // permutohedral_cpu.h:681
    ls->NT = b.NT;
    ls->B = b.B;
    ls->Lmax = Lmax;
    const long long vcap = ((long long)b.NT + b.B) * ls->D;
    if (vcap > INT_MAX / 2) {
        delete ls;
        return fail(LCCRF_ERR_ARG, "batch too large: (NT + B) * (d+1) must stay below 2^30");
    }
    ls->Vcap = (int)((vcap + 1) & ~1LL);  // even: the D neighbour tables [D][Vcap] int2 start at 16-byte multiples (bulk copies)
    const size_t nent = (size_t)(b.NT > 0 ? b.NT : 1) * ls->D;
    int rc = LCCRF_OK;
    rc |= dev_alloc(ctx, (void **)&ls->offset, nent * sizeof(int));
    rc |= dev_alloc(ctx, (void **)&ls->bary, nent * sizeof(float));
    rc |= dev_alloc(ctx, (void **)&ls->nbr, (size_t)ls->D * ls->Vcap * sizeof(int2));
    rc |= dev_alloc(ctx, (void **)&ls->vert_slot, (size_t)ls->Vcap * sizeof(int));
    rc |= dev_alloc(ctx, (void **)&ls->vert_prob, (size_t)ls->Vcap * sizeof(int));
    rc |= dev_alloc(ctx, (void **)&ls->vbase, (size_t)(b.B + 1) * sizeof(int));
    rc |= dev_alloc(ctx, (void **)&ls->norm, (size_t)(b.NT > 0 ? b.NT : 1) * sizeof(float));
    if (Lmax > 0) {
        rc |= dev_alloc(ctx, (void **)&ls->valA, (size_t)ls->Vcap * Lmax * sizeof(float));
        rc |= dev_alloc(ctx, (void **)&ls->valB, (size_t)ls->Vcap * Lmax * sizeof(float));
    }
    rc |= dev_alloc(ctx, (void **)&ls->tab_base, (size_t)(b.B + 1) * sizeof(int));
    {
        const long long E = (long long)b.NT * ls->D;
        const size_t mc = (size_t)(E / kScanChunk + E / kLongRow) + 1;
        if (Lmax > 0) {
            rc |= dev_alloc(ctx, (void **)&ls->chunk_sum, mc * Lmax * sizeof(unsigned long long), true);
            rc |= dev_alloc(ctx, (void **)&ls->chunk_rec, mc * Lmax * kChunkRecBytes);
        }
    }
    if (rc != LCCRF_OK) {
        lattice_set_destroy(ctx, ls);
        return LCCRF_ERR_CUDA;
    }
    // per-problem hash regions: power-of-two size >= 2 * ceil4(N_b) * D  (load factor <= 0.5)
    std::vector<int> tab_base(b.B + 1);
    long long slots = 0;
    for (int i = 0; i < b.B; i++) {
        tab_base[i] = (int)slots;
        long long nb = b.h_prob_ptr[i + 1] - b.h_prob_ptr[i];
        long long need = 2 * ((nb + 3) / 4 * 4) * ls->D;
        long long sz = 64;
        while (sz < need) sz <<= 1;
        slots += sz;
        if (slots > INT_MAX) {
            lattice_set_destroy(ctx, ls);
            return fail(LCCRF_ERR_ARG, "hash table would exceed 2^31 slots");
        }
    }
    tab_base[b.B] = (int)slots;
    ls->tab_slots = slots;
    cudaError_t e = cudaMemcpyAsync(ls->tab_base, tab_base.data(), (size_t)(b.B + 1) * sizeof(int),
                                    cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // tab_base is a stack-lifetime vector
    if (e != cudaSuccess) {
        lattice_set_destroy(ctx, ls);
        return fail(LCCRF_ERR_CUDA, std::string("tab_base upload: ") + cudaGetErrorString(e));
    }
    if (csr_create(ctx, b, ls) != LCCRF_OK) {
        lattice_set_destroy(ctx, ls);
        return LCCRF_ERR_CUDA;
    }
    *out = ls;
    return LCCRF_OK;
}

int lattice_set_ensure_L(Ctx *ctx, LatticeSet *ls, int L) {
    if (L <= ls->Lmax) return LCCRF_OK;
    if (L > LCCRF_MAX_L) return fail(LCCRF_ERR_ARG, "label count exceeds LCCRF_MAX_L");
    dev_free(ctx, ls->valA);
    dev_free(ctx, ls->valB);
    dev_free(ctx, ls->chunk_sum);
    dev_free(ctx, ls->chunk_rec);
    dev_free(ctx, ls->tile_part);
    ls->valA = ls->valB = nullptr;
    ls->chunk_sum = nullptr;
    ls->chunk_rec = nullptr;
    ls->tile_part = nullptr;
    ls->Lmax = 0;
    int rc = LCCRF_OK;
    {
        const size_t mc = (size_t)ls->max_chunks + 1;
        rc |= dev_alloc(ctx, (void **)&ls->chunk_sum, mc * L * sizeof(unsigned long long), true);
        rc |= dev_alloc(ctx, (void **)&ls->chunk_rec, mc * L * kChunkRecBytes);
    }
    rc |= dev_alloc(ctx, (void **)&ls->valA, (size_t)ls->Vcap * L * sizeof(float));
    rc |= dev_alloc(ctx, (void **)&ls->valB, (size_t)ls->Vcap * L * sizeof(float));
    rc |= dev_alloc(ctx, (void **)&ls->tile_part, ((size_t)ls->n_tiles + 1) * L * sizeof(float));
    if (rc != LCCRF_OK) return LCCRF_ERR_CUDA;
    ls->Lmax = L;
    return LCCRF_OK;
}

void lattice_set_destroy(Ctx *ctx, LatticeSet *ls) {
    if (!ls) return;
    dev_free(ctx, ls->offset);
    dev_free(ctx, ls->bary);
    dev_free(ctx, ls->nbr);
    dev_free(ctx, ls->vert_slot);
    dev_free(ctx, ls->vert_prob);
    dev_free(ctx, ls->vbase);
    dev_free(ctx, ls->norm);
    dev_free(ctx, ls->valA);
    dev_free(ctx, ls->valB);
    dev_free(ctx, ls->tab_base);
    csr_destroy(ctx, ls);
    delete ls;
}

namespace {

// hash scratch, build kernels up to k_hash_clear
int build_enqueue(Ctx *ctx, const Batch &b, LatticeSet *ls, const float *feat_dev, Ctx::BuildScratch &bs, bool dirty) {
    const int d = ls->d, D = ls->D;
    const long long slots = ls->tab_slots;
    const int NLEV = num_levels(d);
    auto hash_region = [&](Ctx::Scratch &s, size_t bytes, int fill) -> int {
        const size_t had = s.p ? s.bytes : 0;  // ctx_scratch changes the size whenever it allocates
        LCCRF_TRY(ctx_scratch(ctx, s, bytes));
        if (s.bytes != had || dirty) LCCRF_CUDA(cudaMemsetAsync(s.p, fill, s.bytes, ctx->stream));
        return LCCRF_OK;
    };
    for (int lev = 0; lev < NLEV; lev++) LCCRF_TRY(hash_region(bs.hash_keys[lev], (size_t)slots * sizeof(uint64_t), 0));
    LCCRF_TRY(hash_region(bs.hash_first, (size_t)slots * sizeof(int), 0x7f));
    if (dirty) {  // levels this build does not use may hold keys of a deeper lattice's failed build
        for (int lev = NLEV; lev < 3; lev++)
            if (bs.hash_keys[lev].p) LCCRF_CUDA(cudaMemsetAsync(bs.hash_keys[lev].p, 0, bs.hash_keys[lev].bytes, ctx->stream));
    }
    LCCRF_TRY(ctx_scratch(ctx, bs.hash_id, (size_t)slots * sizeof(int)));
    const long long S = ((long long)b.NT + b.B) * D;
    LCCRF_TRY(ctx_scratch(ctx, bs.ent_slot, (size_t)S * sizeof(int)));
    const long long ntiles = S > 0 ? cdiv(S, kIdTile) : 1;
    LCCRF_TRY(ctx_scratch(ctx, bs.ids_status, (size_t)(ntiles + 1) * sizeof(unsigned long long)));

    BuildParams p;
    memset(&p, 0, sizeof(p));
    p.NT = b.NT;
    p.B = b.B;
    p.prob_ptr = b.prob_ptr;
    p.tab_base = ls->tab_base;
    p.feat = feat_dev;
    for (int lev = 0; lev < NLEV; lev++) p.key[lev] = (uint64_t *)bs.hash_keys[lev].p;
    p.first = (int *)bs.hash_first.p;
    p.tab_id = (int *)bs.hash_id.p;
    p.ent_slot = (int *)bs.ent_slot.p;
    p.bary = ls->bary;
    p.offset = ls->offset;
    p.nbr = ls->nbr;
    p.vert_slot = ls->vert_slot;
    p.vert_prob = ls->vert_prob;
    p.vbase = ls->vbase;
    p.Vcap = ls->Vcap;
    p.status = ctx->d_status;
    // constants in double, rounded once (permutohedral_cpu.h:282-285)
    float inv_std_dev = (float)(sqrt(2.0 / 3.0) * (d + 1));
    for (int i = 0; i < d; i++) p.scale[i] = (float)(1.0 / sqrt((double)((i + 2) * (i + 1))) * (double)inv_std_dev);
    p.invD = 1.0f / (d + 1);
    p.fD = (float)(d + 1);
    unsigned long long *ids_status = (unsigned long long *)bs.ids_status.p;
    int rc = LCCRF_ERR_ARG;
    switch (d) {
        case 1: rc = launch_build<1>(ctx, p, ids_status); break;
        case 2: rc = launch_build<2>(ctx, p, ids_status); break;
        case 3: rc = launch_build<3>(ctx, p, ids_status); break;
        case 4: rc = launch_build<4>(ctx, p, ids_status); break;
        case 5: rc = launch_build<5>(ctx, p, ids_status); break;
        case 6: rc = launch_build<6>(ctx, p, ids_status); break;
        case 7: rc = launch_build<7>(ctx, p, ids_status); break;
        default: return fail(LCCRF_ERR_ARG, "unsupported feature dimension");
    }
    return rc;
}

}  // namespace

__global__ void k_hash_in_use(const uint64_t *key, const int *first, long long n, unsigned long long *count) {
    unsigned long long c = 0;
    for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads)
        c += (key && key[i] != 0ull) || (first && first[i] != 0x7f7f7f7f);
    if (c) atomicAdd(count, c);
}

int build_scratch_in_use(Ctx *ctx, long long *slots) {
    unsigned long long *d_count = nullptr, h_count = 0;
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->aux_stream) LCCRF_CUDA(cudaStreamSynchronize(ctx->aux_stream));
    LCCRF_CUDA(cudaMalloc(&d_count, sizeof(unsigned long long)));
    cudaError_t e = cudaMemset(d_count, 0, sizeof(unsigned long long));
    for (const Ctx::BuildScratch &bs : ctx->bs) {
        for (const Ctx::Scratch &k : bs.hash_keys)
            if (e == cudaSuccess && k.p) {
                k_hash_in_use<<<persistent_grid((long long)(k.bytes / 8), kThreads, 4), kThreads>>>((const uint64_t *)k.p, nullptr, (long long)(k.bytes / 8), d_count);
                e = cudaGetLastError();
            }
        if (e == cudaSuccess && bs.hash_first.p) {
            k_hash_in_use<<<persistent_grid((long long)(bs.hash_first.bytes / 4), kThreads, 4), kThreads>>>(nullptr, (const int *)bs.hash_first.p, (long long)(bs.hash_first.bytes / 4), d_count);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaMemcpy(&h_count, d_count, sizeof(h_count), cudaMemcpyDeviceToHost);
    cudaFree(d_count);
    if (e != cudaSuccess) return fail(LCCRF_ERR_CUDA, std::string("build_scratch_in_use: ") + cudaGetErrorString(e));
    *slots = (long long)h_count;
    return LCCRF_OK;
}

int lattice_set_build(Ctx *ctx, const Batch &b, LatticeSet *ls, const float *feat_dev) {
    Ctx::BuildScratch &bs = ctx->bs[ctx->branch];
    // Between builds every hash region is empty (keys 0, first 0x7f7f7f7f): a build empties the slots it used
    // (k_hash_clear), so only a freshly allocated buffer, or every buffer after a build that stopped before its clear,
    // is cleared in full.  The scratch counts as dirty from here until k_hash_clear is enqueued.
    const bool dirty = bs.hash_dirty;
    bs.hash_dirty = true;
    const int rc = build_enqueue(ctx, b, ls, feat_dev, bs, dirty);
    if (rc != LCCRF_OK) {
        ctx->scratch_gen++;  // captured graphs of other objects have no clear in front of their builds: drop them
        return rc;
    }
    bs.hash_dirty = false;
    return csr_build(ctx, b, ls);
}

}  // namespace lccrf
