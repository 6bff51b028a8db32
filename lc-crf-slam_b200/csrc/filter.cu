// filter.cu -- splat / blur / slice over a batch of permutohedral lattices.
// Replaces PermutohedralLatticeCPU::compute (Thirdparty/DenseCRF/include/permutohedral_cpu.h:634-699).
//
//   k_splat   (:653-661)  values[v] += bary * in[i]  as a segmented reduction over the vertex-sorted
//             entries of csr.cu, each row summed in point order: no atomics, bit-exact with the
//             reference's sequential float accumulation.
//   k_blur    (:663-679)  new[v] = old[v] + 0.5*(old[n1] + old[n2]), one pass per lattice axis,
//             coalesced over [vertex][label].
//   k_slice   (:684-694)  out[i] = sum_r (bary*alpha) * values[v_r]  (association of the SSE overload).
// The mean-field update fuses PottsPotential3D::apply (pairwise3d.h:73-78) into the slice.
#include <cfloat>
#include <climits>

#include "engine.cuh"

namespace lccrf {

namespace {

// ---------------------------------------------------------------- splat
// Segmented reduction over the vertex-sorted entries (csr.cu).  values[v][l] = (((0 + w0*x0) + w1*x1) + ...)
// over the row of v in point order, every product and sum individually rounded -- the reference's splat loop
// (:653-661) bit for bit.  The kernels gather in[point] themselves (no intermediate product array):
//   k_splat_rows                 rows shorter than kLongRow, by tiles of kTreeTile sorted entries (further down)
//   k_scan_compose, k_scan_walk  rows of kLongRow entries and more: exact parallel scan (next section)
//   k_splat_tree, k_splat_carry  tolerance mode (option "ordered_splat" = 0): fixed-shape tree per row

// labels staged per pass
static inline int tile_labels(int L) { return L <= 2 ? L : 4; }

// ---------------------------------------------------------------- exact ordered scan for long rows
// A lane-sequential walk costs one dependent FADD (4 cycles) plus load latency per entry, which is too slow for
// rows with thousands of entries.  The sequential fp32 sum s <- RN(s + c_k) can nevertheless be evaluated in
// parallel EXACTLY: while s stays inside one binade [2^E, 2^(E+1)) its ulp u = 2^(E-23) is constant, s = m*u with
// an integer m, and RN(s + c) = (m + n + r)*u where c/u = n + f (n = floor) and r = [f > 1/2], or, on a tie
// f == 1/2, whatever makes the result even (round-half-even).  "m -> m + a_parity(m)" maps compose
// associatively as pairs (a_even, a_odd), so a block of entries is an inclusive scan of such pairs.  The first
// entry whose prefix leaves the binade is added with one real FADD and the scan restarts behind it; a row of
// 100k entries needs ~17 restarts.  Verified against sequential summation incl. ties, signs, zeros and jumps.
struct ScanPair {
    int a0, a1;
};
__device__ __forceinline__ ScanPair scan_combine(ScanPair l, ScanPair r) {  // apply l first, then r
    ScanPair o;
    o.a0 = l.a0 + ((l.a0 & 1) ? r.a1 : r.a0);
    o.a1 = l.a1 + ((l.a1 & 1) ? r.a0 : r.a1);
    return o;
}

// One product in ulps of the binade, q = c/u (a power-of-two scaling: exact unless it underflows, far below 1/2), split as n = floor(q) and its fraction
// against 1/2: up = fraction > 1/2, tie = fraction == 1/2.  Read from floor(2q), which is exact; q - floor(q) is not
// for -1/2 < q < 0, where q = -1/2 + 2^-25 would round to a fraction of exactly 1/2 and pass for a tie.
// |q| >= 2^24, inf and NaN give n = +-2^24, which no safe range admits.  NONNEG: q >= 0 (a monotone chunk), where
// q - floor(q) is exact and costs less.
template <bool NONNEG = false>
__device__ __forceinline__ void split_ulps(float q, int &n, bool &up, bool &tie) {
    up = tie = false;
    if (!(fabsf(q) < 16777216.0f)) {
        n = q > 0.0f ? (1 << 24) : -(1 << 24);
        return;
    }
    if (NONNEG) {
        n = __float2int_rd(q);
        const float fr = __fsub_rn(q, (float)n);
        up = fr > 0.5f;
        tie = fr == 0.5f;
        return;
    }
    const float q2 = __fmul_rn(q, 2.0f);
    const int i2 = __float2int_rd(q2);
    n = i2 >> 1;
    if (i2 & 1) {
        tie = __int2float_rn(i2) == q2;
        up = !tie;
    }
}

// The increments are rounded on the grid of binade E, which is only the true grid while the exact running sum stays
// in [2^E, 2^(E+1)).  Below 2^E the grid is twice as fine, so an exact sum in [2^E - u/2, 2^E - u/4) rounds to 2^E on
// E's grid but not in fp32.  The lower bound of a safe range is therefore taken over the exact prefixes: an entry
// contributes (its rounded prefix in front of it) + floor(q), below which the exact sum behind it cannot lie.

template <int NW>
struct ScanShared {
    ScanPair warp_tot[NW > 1 ? NW : 1];
    int first_bad[NW > 1 ? NW : 1];
    float bcast[2];
};

// barrier of a team of NW warps (named barrier 1: sub-teams of a CTA may run it while the other warps wait at barrier 0)
template <int NW>
__device__ __forceinline__ void team_sync() {
    if (NW > 1) asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
}

// Exact sequential sum s0 + c[e0] + c[e0+1] + ... (c = bary * in[point], label l) over the entries [e0, e1), computed
// by a team of NW warps; every thread owns IT consecutive entries of each chunk of NW*32*IT.  All threads of the team
// call this with identical arguments; tid = thread index inside the team.  Returns the same value in every thread.
template <int NW, int IT>
__device__ float row_sum_exact(const int2 *__restrict__ ent, const float *__restrict__ in, int e0, int e1, int L, int l,
                               int tid, ScanShared<NW> &sh, float s) {
    constexpr int T = NW * 32, CH = T * IT;
    const int lane = tid & 31, wid = tid >> 5;
    const float *x = in + l;
    // software pipeline over chunks: (wn, xn) = weights and gathered values of the next chunk, en = entries of the
    // chunk after it; both are in flight while the current chunk is scanned (the multiply happens at consumption,
    // so no instruction waits on a load before the scan work)
    float wn[IT], xn[IT];
    int2 en[IT];
#pragma unroll
    for (int k = 0; k < IT; k++) en[k] = e0 + tid * IT + k < e1 ? __ldg(ent + e0 + tid * IT + k) : make_int2(0, 0);
#pragma unroll
    for (int k = 0; k < IT; k++) {
        wn[k] = __int_as_float(en[k].y);
        xn[k] = e0 + tid * IT + k < e1 ? __ldg(x + (size_t)en[k].x * L) : 0.0f;
    }
#pragma unroll
    for (int k = 0; k < IT; k++)
        en[k] = e0 + CH + tid * IT + k < e1 ? __ldg(ent + e0 + CH + tid * IT + k) : make_int2(0, 0);
    for (int cb = e0; cb < e1; cb += CH) {
        float c[IT];
#pragma unroll
        for (int k = 0; k < IT; k++) c[k] = __fmul_rn(wn[k], xn[k]);
        {
            const int nbase = cb + CH + tid * IT;
#pragma unroll
            for (int k = 0; k < IT; k++) {
                wn[k] = __int_as_float(en[k].y);
                xn[k] = nbase + k < e1 ? __ldg(x + (size_t)en[k].x * L) : 0.0f;
            }
#pragma unroll
            for (int k = 0; k < IT; k++) en[k] = nbase + CH + k < e1 ? __ldg(ent + nbase + CH + k) : make_int2(0, 0);
        }
        const int n_chunk = min(CH, e1 - cb);
        const int li0 = tid * IT;  // chunk-local index of this thread's first entry
        int st = 0;                // entries [0, st) of the chunk are already folded into s
        while (st < n_chunk) {
            const int E = ((__float_as_int(s) >> 23) & 0xff) - 127;
            const bool regular = (s > 0.0f) && E >= -100 && E <= 100;
            if (!regular) {
                // rare path (row start, zero / negative / huge running sums): one real addition at a time,
                // except that a run of exact zeros is skipped while s == +0
                team_sync<NW>();
                if (s == 0.0f) {
                    int first = CH;
#pragma unroll
                    for (int k = IT - 1; k >= 0; k--)
                        if (li0 + k >= st && li0 + k < n_chunk && c[k] != 0.0f) first = li0 + k;
#pragma unroll
                    for (int o = 16; o; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
                    if (NW > 1) {
                        if (lane == 0) sh.first_bad[wid] = first;
                        team_sync<NW>();
                        first = CH;
#pragma unroll
                        for (int w = 0; w < NW; w++) first = min(first, sh.first_bad[w]);
                        team_sync<NW>();
                    }
                    if (first >= n_chunk) {
                        st = n_chunk;
                        continue;
                    }
                    st = first;
                }
                float cj = 0.0f;
#pragma unroll
                for (int k = 0; k < IT; k++)
                    if (li0 + k == st) cj = c[k];
                if (NW == 1) cj = __shfl_sync(0xffffffffu, cj, st / IT);
                else {
                    if (tid == st / IT) sh.bcast[1] = cj;
                    team_sync<NW>();
                    cj = sh.bcast[1];
                }
                s = __fadd_rn(s, cj);
                st++;
                continue;
            }
            const float u = __int_as_float((E - 23 + 127) << 23);
            const float inv_u = __int_as_float((23 - E + 127) << 23);
            const int m0 = (int)__fmul_rn(s, inv_u);  // in [2^23, 2^24)
            // thread-local composition of this thread's entries + excursion bounds for either start parity
            ScanPair tot;
            tot.a0 = tot.a1 = 0;
            int hi0 = 0, lo0 = 0, hi1 = 0, lo1 = 0;
            if (li0 + IT > st && li0 < n_chunk) {  // threads whose entries are already folded in contribute the identity
#pragma unroll
                for (int k = 0; k < IT; k++) {
                    if (li0 + k >= st && li0 + k < n_chunk) {
                        int ni;
                        bool up, tie;
                        split_ulps(__fmul_rn(c[k], inv_u), ni, up, tie);
                        lo0 = min(lo0, tot.a0 + ni);  // floor of the exact prefix behind this entry
                        lo1 = min(lo1, tot.a1 + ni);
                        if (!tie) {  // common case: the same increment for either parity
                            const int inc1 = ni + (up ? 1 : 0);
                            tot.a0 += inc1;
                            tot.a1 += inc1;
                        } else {     // tie: round half to even
                            ScanPair a;
                            a.a0 = ni + (ni & 1);
                            a.a1 = ni + ((ni + 1) & 1);
                            tot = scan_combine(tot, a);
                        }
                        hi0 = max(hi0, tot.a0);
                        hi1 = max(hi1, tot.a1);
                    }
                }
            }
            // exclusive scan of the thread totals in thread order
            ScanPair inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                ScanPair lft;
                lft.a0 = __shfl_up_sync(0xffffffffu, inc.a0, o);
                lft.a1 = __shfl_up_sync(0xffffffffu, inc.a1, o);
                if (lane >= o) inc = scan_combine(lft, inc);
            }
            ScanPair exc;
            exc.a0 = __shfl_up_sync(0xffffffffu, inc.a0, 1);
            exc.a1 = __shfl_up_sync(0xffffffffu, inc.a1, 1);
            if (lane == 0) exc.a0 = exc.a1 = 0;
            if (NW > 1) {
                if (lane == 31) sh.warp_tot[wid] = inc;
                team_sync<NW>();
                // every warp scans the NW warp totals itself (no second barrier)
                ScanPair w = sh.warp_tot[lane < NW ? lane : 0];
                if (lane >= NW) w.a0 = w.a1 = 0;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    ScanPair lft;
                    lft.a0 = __shfl_up_sync(0xffffffffu, w.a0, o);
                    lft.a1 = __shfl_up_sync(0xffffffffu, w.a1, o);
                    if (lane >= o) w = scan_combine(lft, w);
                }
                ScanPair wp;  // composite of all warps before this one
                wp.a0 = __shfl_sync(0xffffffffu, w.a0, wid > 0 ? wid - 1 : 0);
                wp.a1 = __shfl_sync(0xffffffffu, w.a1, wid > 0 ? wid - 1 : 0);
                if (wid > 0) exc = scan_combine(wp, exc);
            }
            const int m_start = m0 + ((m0 & 1) ? exc.a1 : exc.a0);
            const int hi = (m_start & 1) ? hi1 : hi0, lo = (m_start & 1) ? lo1 : lo0;
            const bool ok = (m_start + lo >= (1 << 23)) && (m_start + hi < (1 << 24));
            const int m_end = m_start + ((m_start & 1) ? tot.a1 : tot.a0);
            const unsigned badmask = __ballot_sync(0xffffffffu, !ok);
            int tb;  // first thread whose entries leave the binade
            if (NW == 1) {
                tb = badmask ? __ffs(badmask) - 1 : T;
            } else {
                if (lane == 0) sh.first_bad[wid] = badmask ? wid * 32 + __ffs(badmask) - 1 : T;
                if (tid == T - 1) sh.bcast[0] = __fmul_rn((float)m_end, u);
                team_sync<NW>();
                tb = T;
#pragma unroll
                for (int w = NW - 1; w >= 0; w--) {
                    const int fb = sh.first_bad[w];
                    if (fb < T) tb = fb;
                }
            }
            if (tb == T) {  // the rest of the chunk stayed inside the binade
                if (NW == 1) s = __shfl_sync(0xffffffffu, __fmul_rn((float)m_end, u), 31);
                else s = sh.bcast[0];
                st = n_chunk;
            } else {  // threads before tb are consumed by the scan; thread tb adds its entries for real
                float sq = __fmul_rn((float)m_start, u);
                if (tid == tb) {
#pragma unroll
                    for (int k = 0; k < IT; k++)
                        if (li0 + k >= st && li0 + k < n_chunk) sq = __fadd_rn(sq, c[k]);
                }
                if (NW == 1) s = __shfl_sync(0xffffffffu, sq, tb);
                else {
                    if (tid == tb) sh.bcast[1] = sq;
                    team_sync<NW>();
                    s = sh.bcast[1];
                }
                st = min((tb + 1) * IT, n_chunk);
            }
            // shared words written above are rewritten only after the next team barrier of this loop
        }
    }
    return s;
}

// ---------------------------------------------------------------- long rows: speculative parallel scan
// A row of 67k entries is still one dependent chain if a single CTA walks it chunk by chunk.  But inside a binade
// the effect of a whole chunk on the running sum is the pair composite (a_even, a_odd) -- it depends on the running
// sum only through its binade (the ulp) and its parity.  The binade at the start of every chunk is predictable from
// plain (unordered) chunk sums, so ALL chunks of ALL long rows are composed in parallel, and the sequential part
// shrinks to one O(1) step per chunk:
//   k_scan_compose  per (chunk, label), one WARP per task: unordered fp32 sum of the chunk's products, published to the
//                   chunks behind it; predicted start sum -> binade E; composite (a0, a1) of the chunk under that
//                   binade and the range of start values for which no prefix leaves the binade (parallel); the row
//                   heads (start value +0) are summed for real
//   k_scan_walk     per (row, label): walks the chunk records; a record applies iff the true running sum is in
//                   the predicted binade and inside the record's safe range -- then s <- (m + a_parity) * ulp,
//                   exactly what the entry-by-entry additions would give.  Otherwise (the chunk that contains a
//                   binade crossing, a mispredicted binade, the row head) the chunk is summed for real with
//                   row_sum_exact.  Either way the result is the sequential fp32 sum, bit for bit.
// One record per (chunk, label).  kind:
//   kRecNone   no composite (irregular prediction): the walk sums the chunk for real
//   kRecExact  s_exact = the exact running sum at the END of the chunk (row heads: the start value 0 is known)
//   kRecPlain  composite A covers the whole chunk under binade E
//   kRecCross  the running sum is predicted to cross from binade E to E+1 inside the chunk: composite A covers the
//              entries before the crossing window (binade E), win[] holds the products of the window (32 entries,
//              added for real by the walk), composite B covers the entries behind it (binade E+1)
//   kRecZero   every product of the chunk is +-0: the chunk leaves any running sum unchanged (a row start is +0 and a
//              running sum never becomes -0, so adding +-0 is the identity) -- typical for a label whose marginal
//              hit the fast_exp cut-off on all points of a vertex
enum { kRecNone = 0, kRecExact = 1, kRecPlain = 2, kRecCross = 3, kRecZero = 4 };
constexpr int kWinThreads = 4;                     // lanes (of 8 entries each) covered by the crossing window
struct Composite {
    int a0, a1;              // total increment in ulps for an even / odd start mantissa
    int lo0, hi0, lo1, hi1;  // extreme prefix increments for an even / odd start
};
struct ChunkRec {
    int kind;
    int E;            // predicted binade (unbiased exponent of the running sum) at the start of the chunk
    float s_exact;
    int pad;
    Composite A, B;
    float win[kWinThreads * (kScanChunk / 256)];
};

static_assert(sizeof(ChunkRec) == kChunkRecBytes, "engine.cuh: kChunkRecBytes must match ChunkRec");

// chunk descriptor (csr.cu: k_long_chunks): {first entry, one past the last entry, index of the row's first chunk,
// index of the row in the long list}
constexpr int kScanIT = kScanChunk / 256;  // entries per lane and round (a warp walks a chunk in rounds of 256 entries)

// labels handled per (chunk, label-group) task: the float2 of a point serves both labels of the SLAM CRF
static inline int scan_labels(int L) { return L >= 2 ? 2 : 1; }

template <int LG>
__device__ __forceinline__ void gather_labels(const float *__restrict__ in, int pt, int L, int lb, bool valid, float (&x)[LG]) {
    if (LG == 2 && L == 2) {
        const float2 v = valid ? __ldg((const float2 *)in + pt) : make_float2(0.f, 0.f);
        x[0] = v.x;
        x[LG - 1] = v.y;
    } else {
#pragma unroll
        for (int j = 0; j < LG; j++) x[j] = (valid && lb + j < L) ? __ldg(in + (size_t)pt * L + lb + j) : 0.0f;
    }
}

// per-thread composite of the products c[0..IT) under the binade with ulp 1/inv_u (same arithmetic as row_sum_exact)
template <int IT, bool MONO>
__device__ __forceinline__ void thread_composite(const float *c, int n_valid, float inv_u, ScanPair &tot, int &hi0,
                                                 int &lo0, int &hi1, int &lo1, bool &tie) {
    tot.a0 = tot.a1 = 0;
    hi0 = lo0 = hi1 = lo1 = 0;
    tie = false;
#pragma unroll
    for (int q = 0; q < IT; q++) {
        if (q < n_valid) {
            int ni;
            bool up, t;
            split_ulps<MONO>(__fmul_rn(c[q], inv_u), ni, up, t);
            if (!MONO) {  // floor of the exact prefix behind this entry
                lo0 = min(lo0, tot.a0 + ni);
                lo1 = min(lo1, tot.a1 + ni);
            }
            if (!t) {  // common case: the same increment for either parity
                const int inc1 = ni + (up ? 1 : 0);
                tot.a0 += inc1;
                tot.a1 += inc1;
            } else {   // tie: round half to even
                tie = true;
                ScanPair a;
                a.a0 = ni + (ni & 1);
                a.a1 = ni + ((ni + 1) & 1);
                tot = scan_combine(tot, a);
            }
            if (!MONO) {
                hi0 = max(hi0, tot.a0);
                hi1 = max(hi1, tot.a1);
            }
        }
    }
}

// ---- composites: one warp owns a (chunk, label group) task and walks the chunk in rounds of 256 entries (lane-contiguous,
// 8 entries per lane and round); nothing needs a CTA barrier.  (Round 1 and most of round 2 ran one CTA per chunk with
// block-wide scans: the same instruction count, but barrier-coupled; this form is 1.5 % faster per step beside the other
// stream's kernels.)
//   phase 1 (tickets counts[9]): unordered sum + "has a negative product" / "all products are +-0" flags of every chunk,
//            published as ONE 64-bit word {call tag, flags, sum} (st.relaxed.gpu); all-zero chunks get their kRecZero
//            record right here
//   heads   (static, first CTAs): the first chunk of every long row, summed for real
//   phase 2 (tickets counts[3]): composites; the prediction polls (ld.relaxed.gpu) the words of the chunks in front
// Tickets are taken by running warps only and a word is published without waiting for anything, so a polling warp only
// ever waits for warps that are running -- no residency assumption.  k_scan_walk clears the words it has walked and
// bumps the tag behind every compose launch, so a word is 0 or belongs to the launch that is running.
constexpr unsigned kPubNeg = 2u, kPubZero = 1u;
__device__ __forceinline__ void publish_word(unsigned long long *p, unsigned tag, unsigned flags, float sum) {
    const unsigned long long w = ((unsigned long long)((tag << 2) | flags) << 32) | (unsigned long long)__float_as_uint(sum);
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
__device__ __forceinline__ float poll_word(const unsigned long long *p, unsigned tag, unsigned &flags) {
    unsigned long long w;
    for (;;) {
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
        if ((unsigned)(w >> 34) == tag) break;
        __nanosleep(64);
    }
    flags = (unsigned)(w >> 32) & 3u;
    return __uint_as_float((unsigned)w);
}

// composite of the lanes with `active` of one round (uniform result): total increments for an even / odd start and the
// extreme prefix increments.  tie_any (uniform): some lane met a round-half-even tie, i.e. a0 != a1 somewhere.
template <bool MONO>
__device__ __forceinline__ Composite warp_round_composite(ScanPair tot, int hi0, int lo0, int hi1, int lo1, bool active,
                                                          bool tie_any, int lane) {
    Composite c;
    if (!active) {
        tot.a0 = tot.a1 = 0;
        hi0 = lo0 = hi1 = lo1 = 0;
    }
    if (MONO && !tie_any) {  // plain sum of the increments
        const int sm = __reduce_add_sync(0xffffffffu, tot.a0);
        c.a0 = c.a1 = c.hi0 = c.hi1 = sm;
        c.lo0 = c.lo1 = 0;
        return c;
    }
    ScanPair inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        ScanPair lft;
        lft.a0 = __shfl_up_sync(0xffffffffu, inc.a0, o);
        lft.a1 = __shfl_up_sync(0xffffffffu, inc.a1, o);
        if (lane >= o) inc = scan_combine(lft, inc);
    }
    c.a0 = __shfl_sync(0xffffffffu, inc.a0, 31);
    c.a1 = __shfl_sync(0xffffffffu, inc.a1, 31);
    if (MONO) {
        c.lo0 = c.lo1 = 0;
        c.hi0 = c.a0;
        c.hi1 = c.a1;
        return c;
    }
    ScanPair exc;
    exc.a0 = __shfl_up_sync(0xffffffffu, inc.a0, 1);
    exc.a1 = __shfl_up_sync(0xffffffffu, inc.a1, 1);
    if (lane == 0) exc.a0 = exc.a1 = 0;
    // for a start of parity p this lane begins at offset exc.a_p with parity (p + exc.a_p) & 1
    int b_lo0 = exc.a0 + ((exc.a0 & 1) ? lo1 : lo0), b_hi0 = exc.a0 + ((exc.a0 & 1) ? hi1 : hi0);
    int b_lo1 = exc.a1 + ((exc.a1 & 1) ? lo0 : lo1), b_hi1 = exc.a1 + ((exc.a1 & 1) ? hi0 : hi1);
    if (!active) {  // identity lanes must not widen the range with offsets of ranges they do not belong to
        b_lo0 = b_lo1 = 0;
        b_hi0 = b_hi1 = 0;
    }
    c.lo0 = min(0, __reduce_min_sync(0xffffffffu, b_lo0));
    c.hi0 = max(0, __reduce_max_sync(0xffffffffu, b_hi0));
    c.lo1 = min(0, __reduce_min_sync(0xffffffffu, b_lo1));
    c.hi1 = max(0, __reduce_max_sync(0xffffffffu, b_hi1));
    return c;
}

// R <- R followed by C (both uniform)
__device__ __forceinline__ void composite_append(Composite &R, const Composite &C) {
    const int o0 = R.a0, o1 = R.a1;
    R.lo0 = min(R.lo0, o0 + ((o0 & 1) ? C.lo1 : C.lo0));
    R.hi0 = max(R.hi0, o0 + ((o0 & 1) ? C.hi1 : C.hi0));
    R.lo1 = min(R.lo1, o1 + ((o1 & 1) ? C.lo0 : C.lo1));
    R.hi1 = max(R.hi1, o1 + ((o1 & 1) ? C.hi0 : C.hi1));
    R.a0 = o0 + ((o0 & 1) ? C.a1 : C.a0);
    R.a1 = o1 + ((o1 & 1) ? C.a0 : C.a1);
}

// state of one label of a phase-2 task (uniform across the warp)
struct LabelTask {
    int kind, E;
    bool mono, crossed;
    float top, inv_u, P;  // 2^(E+1), 1/ulp of binade E, predicted running sum in front of the current round
    Composite A, B;
};

template <bool MONO>
__device__ __forceinline__ void label_round(LabelTask &T, const float (&cq)[kScanIT], int n_valid, int r, int lane,
                                            ChunkRec *__restrict__ rec_out) {
    constexpr int IT = kScanIT;
    // predicted running sum behind this lane's entries of the round
    float lsum = 0.0f;
#pragma unroll
    for (int q = 0; q < IT; q++)
        if (q < n_valid) lsum += cq[q];
    float incl = lsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    const float p_end = T.P + incl;
    T.P += __shfl_sync(0xffffffffu, incl, 31);
    bool inA = !T.crossed, inB = T.crossed;
    int tw = -1;
    if (T.kind == kRecCross && !T.crossed) {  // (uniform)
        // the crossing: the first lane behind whose entries the predicted sum reaches 2^(E+1) (with a small safety margin:
        // the true fp32 running sum differs from the prediction by rounding noise only); the window starts one lane
        // earlier.  A chunk that never gets there keeps its window on the last four lanes of the last round.
        const unsigned hit = __ballot_sync(0xffffffffu, p_end >= T.top * (1.0f - 2e-5f));
        if (hit || r == kScanChunk / 256 - 1) {
            tw = hit ? __ffs(hit) - 2 : 32 - kWinThreads;
            tw = max(0, min(tw, 32 - kWinThreads));
            inA = lane < tw;
            inB = lane >= tw + kWinThreads;
            T.crossed = true;
        }
    }
    ScanPair tot;
    int hi0, lo0, hi1, lo1;
    bool tie;
    thread_composite<IT, MONO>(cq, n_valid, inB ? __fmul_rn(T.inv_u, 0.5f) : T.inv_u, tot, hi0, lo0, hi1, lo1, tie);
    const bool tie_any = __any_sync(0xffffffffu, tie);
    if (tw >= 0) {  // (uniform) the crossing round: lanes before the window -> A, behind it -> B, the window itself is stored
        composite_append(T.A, warp_round_composite<MONO>(tot, hi0, lo0, hi1, lo1, inA, tie_any, lane));
        composite_append(T.B, warp_round_composite<MONO>(tot, hi0, lo0, hi1, lo1, inB, tie_any, lane));
        if (!inA && !inB) {
#pragma unroll
            for (int q = 0; q < IT; q++) rec_out->win[(lane - tw) * IT + q] = q < n_valid ? cq[q] : 0.0f;
        }
    } else if (inB) {  // (uniform)
        composite_append(T.B, warp_round_composite<MONO>(tot, hi0, lo0, hi1, lo1, true, tie_any, lane));
    } else {
        composite_append(T.A, warp_round_composite<MONO>(tot, hi0, lo0, hi1, lo1, true, tie_any, lane));
    }
}

template <int LG>
__global__ void __launch_bounds__(256, 3)
k_scan_compose(const int *__restrict__ row_ptr, const int2 *__restrict__ ent, const float *__restrict__ in,
               const int *__restrict__ list, int *counts, const int *__restrict__ long_chunk0,
               const int4 *__restrict__ chunk_desc, unsigned long long *chunk_sum, ChunkRec *__restrict__ rec, int L) {
    constexpr int IT = kScanIT, NR = kScanChunk / 256;
    __shared__ float s_head[8][256 * LG];
    const int ngrp = (L + LG - 1) / LG;
    const long long n = (long long)counts[1] * ngrp;
    const int nlong = counts[0];
    const unsigned tag = ((unsigned)counts[8] & 0x1fffffffu) + 1u;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // ---- phase 1
    for (;;) {
        long long k = 0;
        if (lane == 0) k = atomicAdd(counts + 9, 1);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= n) break;
        const int c = (int)(k / ngrp), lb = (int)(k % ngrp) * LG;
        const int4 g = __ldg(chunk_desc + c);
        float acc[LG];
        bool zero[LG], neg[LG];
#pragma unroll
        for (int j = 0; j < LG; j++) {
            acc[j] = 0.0f;
            zero[j] = true;
            neg[j] = false;
        }
        for (int e = g.x + lane; e < g.y; e += 32 * 8) {  // eight entries per lane in flight (the loop is latency-bound)
            int2 t[8];
            float x[8][LG];
#pragma unroll
            for (int q = 0; q < 8; q++) t[q] = e + 32 * q < g.y ? __ldg(ent + e + 32 * q) : make_int2(0, 0);
#pragma unroll
            for (int q = 0; q < 8; q++) gather_labels<LG>(in, t[q].x, L, lb, e + 32 * q < g.y, x[q]);
#pragma unroll
            for (int q = 0; q < 8; q++) {
                if (e + 32 * q < g.y) {
#pragma unroll
                    for (int j = 0; j < LG; j++) {
                        const float pr = __fmul_rn(__int_as_float(t[q].y), x[q][j]);
                        acc[j] += pr;
                        zero[j] = zero[j] && pr == 0.0f;
                        neg[j] = neg[j] || !(pr >= 0.0f);  // NaN counts as negative: full tracking
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < LG; j++) {
#pragma unroll
            for (int o = 16; o; o >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
            const bool z = __all_sync(0xffffffffu, zero[j]), ng = __any_sync(0xffffffffu, neg[j]);
            if (lane == 0 && lb + j < L) {
                // every product is +-0: the chunk is the identity (a row head keeps its exact record)
                if (z && c != g.z) rec[(size_t)c * L + lb + j].kind = kRecZero;
                publish_word(chunk_sum + (size_t)c * L + lb + j, tag, (z ? kPubZero : 0u) | (ng ? kPubNeg : 0u), acc[j]);
            }
        }
    }
    // ---- row heads: the start value (+0) is known, so the first chunk of a row is summed for real, front to back, by ONE
    // lane per label: the warp stages the products of a round (256 entries, coalesced) in shared memory, the lane adds
    // them in order -- 4 cycles per entry, 2048 entries in about 5 microseconds.  (A parallel exact scan is slower here:
    // binade crossings are dense at a row start, and every crossing restarts the scan.)  The first CTAs of the grid take
    // the heads, 8 per CTA.
    {
        const long long nheads = (long long)nlong * ngrp;
        for (long long hk = (long long)blockIdx.x * 8 + wid; hk < nheads; hk += (long long)gridDim.x * 8) {
            const int i = (int)(hk / ngrp), lb = (int)(hk % ngrp) * LG;
            const int v = __ldg(list + i);
            const int e0 = __ldg(row_ptr + v), e1 = min(e0 + kScanChunk, __ldg(row_ptr + v + 1));
            float *stage = s_head[wid];
            float sum = 0.0f;
            int2 tn[IT];
            float xn[IT][LG];
#pragma unroll
            for (int q = 0; q < IT; q++) {
                const int e = e0 + lane * IT + q;
                tn[q] = e < e1 ? __ldg(ent + e) : make_int2(0, 0);
            }
#pragma unroll
            for (int q = 0; q < IT; q++) gather_labels<LG>(in, tn[q].x, L, lb, e0 + lane * IT + q < e1, xn[q]);
            for (int r = 0; r < NR && e0 + r * 256 < e1; r++) {
#pragma unroll
                for (int q = 0; q < IT; q++)
#pragma unroll
                    for (int j = 0; j < LG; j++) stage[(lane * IT + q) * LG + j] = __fmul_rn(__int_as_float(tn[q].y), xn[q][j]);
                if (r + 1 < NR) {
#pragma unroll
                    for (int q = 0; q < IT; q++) {
                        const int e = e0 + (r + 1) * 256 + lane * IT + q;
                        tn[q] = e < e1 ? __ldg(ent + e) : make_int2(0, 0);
                    }
#pragma unroll
                    for (int q = 0; q < IT; q++) gather_labels<LG>(in, tn[q].x, L, lb, e0 + (r + 1) * 256 + lane * IT + q < e1, xn[q]);
                }
                __syncwarp();
                const int cnt = min(256, e1 - (e0 + r * 256));
                if (lane < LG) {
                    int i2 = 0;
                    for (; i2 + 8 <= cnt; i2 += 8) {  // eight operands in flight, then the ordered chain
                        float y[8];
#pragma unroll
                        for (int q = 0; q < 8; q++) y[q] = stage[(i2 + q) * LG + lane];
#pragma unroll
                        for (int q = 0; q < 8; q++) sum = __fadd_rn(sum, y[q]);
                    }
                    for (; i2 < cnt; i2++) sum = __fadd_rn(sum, stage[i2 * LG + lane]);
                }
                __syncwarp();
            }
            if (lane < LG && lb + lane < L) {
                const size_t k = (size_t)__ldg(long_chunk0 + i) * L + lb + lane;
                rec[k].kind = kRecExact;
                rec[k].s_exact = sum;
            }
        }
    }
    // ---- phase 2
    for (;;) {
        long long k = 0;
        if (lane == 0) k = atomicAdd(counts + 3, 1);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= n) break;
        const int c = (int)(k / ngrp), lb = (int)(k % ngrp) * LG;
        const int4 g = __ldg(chunk_desc + c);
        if (c == g.z) continue;  // a row head
        LabelTask T[LG];
        bool any_active = false;
#pragma unroll
        for (int j = 0; j < LG; j++) {
            T[j].kind = -1;  // no record to write
            if (lb + j >= L) continue;
            unsigned fl, fdummy;
            const float own = poll_word(chunk_sum + (size_t)c * L + lb + j, tag, fl);
            float sp = 0.0f;
            for (int jj = g.z + lane; jj < c; jj += 32) sp += poll_word(chunk_sum + (size_t)jj * L + lb + j, tag, fdummy);
#pragma unroll
            for (int o = 16; o; o >>= 1) sp += __shfl_xor_sync(0xffffffffu, sp, o);
            if (fl & kPubZero) continue;  // recorded in phase 1
            const float total = sp + own;  // predicted running sum at the end of the chunk
            const int E = ((__float_as_int(sp) >> 23) & 0xff) - 127;
            const bool regular = (sp > 0.0f) && E >= -100 && E <= 100;
            const float top = __int_as_float((E + 1 + 127) << 23);  // 2^(E+1)
            int kind = kRecNone;
            if (regular) {
                if (total < top * (1.0f - 1e-4f)) kind = kRecPlain;
                else if (total < 2.0f * top * (1.0f - 1e-4f)) kind = kRecCross;
            }
            T[j].kind = kind;
            T[j].E = E;
            T[j].mono = !(fl & kPubNeg);
            T[j].crossed = false;
            T[j].top = top;
            T[j].inv_u = __int_as_float((23 - E + 127) << 23);
            T[j].P = sp;
            T[j].A.a0 = T[j].A.a1 = T[j].A.lo0 = T[j].A.hi0 = T[j].A.lo1 = T[j].A.hi1 = 0;
            T[j].B = T[j].A;
            if (kind == kRecNone) {
                if (lane == 0) rec[(size_t)c * L + lb + j].kind = kRecNone;
            } else {
                any_active = true;
            }
        }
        if (!any_active) continue;  // (uniform)
        // rounds of 256 entries, lane-contiguous; the loads of the next round are in flight while this one is composed
        int2 tn[IT];
        float xn[IT][LG];
#pragma unroll
        for (int q = 0; q < IT; q++) {
            const int e = g.x + lane * IT + q;
            tn[q] = e < g.y ? __ldg(ent + e) : make_int2(0, 0);
        }
#pragma unroll
        for (int q = 0; q < IT; q++) gather_labels<LG>(in, tn[q].x, L, lb, g.x + lane * IT + q < g.y, xn[q]);
        for (int r = 0; r < NR; r++) {
            const int e0 = g.x + r * 256 + lane * IT;
            const int n_valid = max(0, min(IT, g.y - e0));
            float cq[LG][IT];
#pragma unroll
            for (int j = 0; j < LG; j++)
#pragma unroll
                for (int q = 0; q < IT; q++) cq[j][q] = __fmul_rn(__int_as_float(tn[q].y), xn[q][j]);
            if (r + 1 < NR) {
#pragma unroll
                for (int q = 0; q < IT; q++) {
                    const int e = e0 + 256 + q;
                    tn[q] = e < g.y ? __ldg(ent + e) : make_int2(0, 0);
                }
#pragma unroll
                for (int q = 0; q < IT; q++) gather_labels<LG>(in, tn[q].x, L, lb, e0 + 256 + q < g.y, xn[q]);
            }
#pragma unroll
            for (int j = 0; j < LG; j++) {
                if (T[j].kind == kRecPlain || T[j].kind == kRecCross) {  // (uniform)
                    ChunkRec *ro = rec + (size_t)c * L + lb + j;
                    if (T[j].mono) label_round<true>(T[j], cq[j], n_valid, r, lane, ro);
                    else label_round<false>(T[j], cq[j], n_valid, r, lane, ro);
                }
            }
        }
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < LG; j++) {
                if (T[j].kind == kRecPlain || T[j].kind == kRecCross) {
                    ChunkRec *ro = rec + (size_t)c * L + lb + j;
                    ro->kind = T[j].kind;
                    ro->E = T[j].E;
                    ro->A = T[j].A;
                    if (T[j].kind == kRecCross) ro->B = T[j].B;
                }
            }
        }
    }
}

constexpr int kWalkBatch = 32;  // chunk records staged per round

__device__ __forceinline__ bool apply_composite(float &s, int E, const Composite &c) {
    const int Es = ((__float_as_int(s) >> 23) & 0xff) - 127;
    if (!((s > 0.0f) && Es == E)) return false;
    const float u = __int_as_float((E - 23 + 127) << 23);
    const float inv_u = __int_as_float((23 - E + 127) << 23);
    const int m0 = (int)__fmul_rn(s, inv_u);  // in [2^23, 2^24)
    const int lo = (m0 & 1) ? c.lo1 : c.lo0, hi = (m0 & 1) ? c.hi1 : c.hi0;
    if (!(m0 + lo >= (1 << 23) && m0 + hi < (1 << 24))) return false;
    s = __fmul_rn((float)(m0 + ((m0 & 1) ? c.a1 : c.a0)), u);
    return true;
}

__global__ void __launch_bounds__(256)
k_scan_walk(const int *__restrict__ row_ptr, const int2 *__restrict__ ent, const float *__restrict__ in,
            float *__restrict__ val, const int *__restrict__ list, int *counts,
            const int *__restrict__ long_chunk0, const ChunkRec *__restrict__ rec, unsigned long long *chunk_sum, int L) {
    __shared__ ScanShared<8> sh;
    __shared__ ChunkRec s_rec[kWalkBatch];
    const long long n = (long long)counts[0] * L;
    int n_fast = 0, n_cross = 0, n_fall = 0, n_zero = 0;  // diagnostics (counts[4..7])
    const int tid = threadIdx.x;
    if (blockIdx.x == 0 && tid == 0) {  // the compose launch in front is over: reset its tickets, retire its tag
        counts[3] = 0;
        counts[9] = 0;
        counts[8] = counts[8] + 1;
    }
    for (long long k = blockIdx.x; k < n; k += gridDim.x) {
        const int i = (int)(k / L), l = (int)(k % L);
        const int v = __ldg(list + i);
        const int e0 = __ldg(row_ptr + v), e1 = __ldg(row_ptr + v + 1);
        const int c0 = __ldg(long_chunk0 + i), nch = __ldg(long_chunk0 + i + 1) - c0;
        float s = 0.0f;
        for (int cb = 0; cb < nch; cb += kWalkBatch) {
            const int nb = min(kWalkBatch, nch - cb);
            __syncthreads();  // previous round's records consumed
            {   // stage the records of this round (word-wise, coalesced)
                constexpr int W = (int)(sizeof(ChunkRec) / 4);
                const int *src = (const int *)rec;
                int *dst = (int *)s_rec;
                for (int w = tid; w < nb * W; w += 256) {
                    const int j = w / W, o = w - j * W;
                    dst[w] = __ldg(src + ((size_t)(c0 + cb + j) * L + l) * W + o);
                }
                // the published word of every walked (chunk, label) is cleared for the next compose launch: a word is
                // either 0 or carries the tag of the launch that is running, whatever the tag counter does
                if (tid < nb) chunk_sum[(size_t)(c0 + cb + tid) * L + l] = 0ull;
            }
            __syncthreads();
            for (int j = 0; j < nb; j++) {
                const ChunkRec &r = s_rec[j];
                bool done = false;
                if (r.kind == kRecExact) {
                    s = r.s_exact;  // row head
                    done = true;
                } else if (r.kind == kRecZero) {
                    done = true;
                    n_zero++;
                } else if (r.kind == kRecPlain) {
                    done = apply_composite(s, r.E, r.A);
                    n_fast += done;
                } else if (r.kind == kRecCross) {
                    float t = s;
                    if (apply_composite(t, r.E, r.A)) {
#pragma unroll 8
                        for (int q = 0; q < kWinThreads * kScanIT; q++) t = __fadd_rn(t, r.win[q]);
                        if (apply_composite(t, r.E + 1, r.B)) {
                            s = t;
                            done = true;
                            n_cross++;
                        }
                    }
                }
                n_fall += !done;
                if (!done) {  // uniform: s and the record are identical in every thread
                    const int a = e0 + (cb + j) * kScanChunk;
                    s = row_sum_exact<8, kScanIT>(ent, in, a, min(a + kScanChunk, e1), L, l, tid, sh, s);
                }
            }
        }
        if (tid == 0) val[(size_t)v * L + l] = s;
    }
    if (tid == 0 && (n_fast | n_cross | n_fall | n_zero)) {
        atomicAdd(counts + 4, n_fast);
        atomicAdd(counts + 5, n_cross);
        atomicAdd(counts + 6, n_fall);
        atomicAdd(counts + 7, n_zero);
    }
}

// ---------------------------------------------------------------- ordered splat, short rows, by entry tiles
// Every row summed front to back, organised by fixed tiles of kTreeTile sorted entries: a CTA owns the short rows that
// START in its tile and stages the tile plus the kLongRow - 1 entries a short row can reach beyond it.  Phase 1: coalesced entry stream, gather in[point], products to shared memory.  Phase 2: row
// ra + i of the tile is walked by thread i -- one FADD chain per (row, label), operands prefetched eight entries ahead so
// that the chain runs at the adder's latency.  No row pointer staging, no atomics; rows >= kLongRow are left to the scan.
constexpr int kRowsThreads = 256;
constexpr int kRowsWin = kTreeTile + kLongRow;             // staged entries per tile (3072)
constexpr int kRowsIT = kRowsWin / kRowsThreads;           // 12 entries per thread in phase 1

template <int LG>
__global__ void __launch_bounds__(kRowsThreads, LG <= 2 ? 6 : 3)
k_splat_rows(const int *__restrict__ row_ptr, const int *__restrict__ tile_row0, const int *__restrict__ tile_own,
             const int2 *__restrict__ ent, const float *__restrict__ in, float *__restrict__ val, int n_tiles, long long E,
             int L, int lb) {
    extern __shared__ float s_rows[];  // [kRowsWin][LG] products
    const int tid = threadIdx.x;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        if (!__ldg(tile_own + t)) continue;  // (uniform) only long rows here: the scan kernels' business
        const long long t0 = (long long)t * kTreeTile;
        const int cnt = (int)min((long long)kRowsWin - 1, E - t0);
        const int ra = __ldg(tile_row0 + t), rb = __ldg(tile_row0 + t + 1);
        // phase 1, in two halves (register budget: 39 registers, 5-6 CTAs per SM keep enough chains in flight; asking for the
        // largest shared-memory carve-out on top of that was measured 1.7x SLOWER -- the gathers do live in L1)
        constexpr int kHalf = kRowsIT / 2;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            int2 e[kHalf];
#pragma unroll
            for (int q = 0; q < kHalf; q++) {
                const int i = (h * kHalf + q) * kRowsThreads + tid;
                e[q] = i < cnt ? __ldg(ent + t0 + i) : make_int2(0, 0);
            }
            float x[kHalf][LG];
#pragma unroll
            for (int q = 0; q < kHalf; q++) {
                const int i = (h * kHalf + q) * kRowsThreads + tid;
                if (LG == 2 && L == 2) {
                    const float2 v = i < cnt ? __ldg((const float2 *)in + e[q].x) : make_float2(0.f, 0.f);
                    x[q][0] = v.x;
                    x[q][LG - 1] = v.y;
                } else {
#pragma unroll
                    for (int j = 0; j < LG; j++) x[q][j] = (i < cnt && lb + j < L) ? __ldg(in + (size_t)e[q].x * L + lb + j) : 0.0f;
                }
            }
#pragma unroll
            for (int q = 0; q < kHalf; q++) {
                const int i = (h * kHalf + q) * kRowsThreads + tid;
                const float w = __int_as_float(e[q].y);
                if (i < cnt) {
#pragma unroll
                    for (int j = 0; j < LG; j++) s_rows[(size_t)i * LG + j] = __fmul_rn(w, x[q][j]);
                }
            }
        }
        __syncthreads();
        // phase 2: rows that start in this tile
        // (a row without entries -- a vertex only phantom points touch -- belongs to the tile its position follows)
        for (int r = (t == 0 ? 0 : ra) + tid; r <= rb; r += kRowsThreads) {
            const long long s = __ldg(row_ptr + r), z = __ldg(row_ptr + r + 1);
            const bool mine = z > s ? (s >= t0 && s < t0 + kTreeTile) : ((s > t0 && s <= t0 + kTreeTile) || (s == 0 && t == 0));
            if (!mine || z - s >= kLongRow) continue;
            const int a = (int)(s - t0), b = (int)(z - t0);
            float acc[LG];
#pragma unroll
            for (int j = 0; j < LG; j++) acc[j] = 0.0f;
            int i = a;
            for (; i + 4 <= b; i += 4) {  // four operands per label in flight, then the ordered chain
                float y[4][LG];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    if (LG == 2) {
                        const float2 v = *(const float2 *)(s_rows + (size_t)(i + q) * 2);
                        y[q][0] = v.x;
                        y[q][LG - 1] = v.y;
                    } else {
#pragma unroll
                        for (int j = 0; j < LG; j++) y[q][j] = s_rows[(size_t)(i + q) * LG + j];
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; q++)
#pragma unroll
                    for (int j = 0; j < LG; j++) acc[j] = __fadd_rn(acc[j], y[q][j]);
            }
            for (; i < b; i++)
#pragma unroll
                for (int j = 0; j < LG; j++) acc[j] = __fadd_rn(acc[j], s_rows[(size_t)i * LG + j]);
#pragma unroll
            for (int j = 0; j < LG; j++)
                if (lb + j < L) val[(size_t)r * L + lb + j] = acc[j];
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- tree splat (option "ordered_splat" = 0)
// The same segmented reduction over the vertex-sorted entries, but every row is summed by a FIXED-SHAPE TREE instead
// of front to back: one streaming pass, balanced whatever the row lengths are, and deterministic (the shape depends on
// row_ptr only).  Marginals agree with the reference within its own sequential rounding error (tests gate 1e-4
// relative, north_star), not bit for bit -- the ordered kernels above stay the default.
//   k_splat_tree   a CTA owns a tile of kTreeTile consecutive entries.  Phase 1: coalesced entry stream, gather
//                  in[point], products to shared memory; row starts that fall into the tile are marked with their row
//                  id.  Phase 2: thread t folds its 8 consecutive products left to right, a segmented scan over the
//                  threads (warp shuffles + one shared level) closes every row that ends inside the tile.  What is
//                  open at the tile's borders goes to tile_part (the part in front of the first row start) and, as a
//                  partial sum, to val[row open at the end].
//   k_splat_carry  rows that span tiles: partial + the leading parts of the following tiles, in tile order; rows without
//                  entries (vertices only phantom points touch) are zeroed.
constexpr int kTreeThreads = 256;
constexpr int kTreeIT = kTreeTile / kTreeThreads;  // 8 consecutive entries per thread
static_assert(kTreeIT == 8, "padding scheme below assumes 8 entries per thread");
__device__ __forceinline__ int tpad(int i) { return i + (i >> 3); }  // one padding slot per thread: conflict-free both ways

template <int LG>
__global__ void __launch_bounds__(kTreeThreads)
k_splat_tree(const int *__restrict__ row_ptr, const int *__restrict__ tile_row0, const int2 *__restrict__ ent,
             const float *__restrict__ in, float *__restrict__ val, float *__restrict__ tile_part,
             int2 *__restrict__ tile_info, int n_tiles, long long E, int L, int lb) {
    __shared__ float s_prod[LG][kTreeTile + kTreeTile / 8];
    __shared__ int s_row[kTreeTile + kTreeTile / 8];   // row id of the row that starts at this entry, -1 otherwise
    __shared__ float s_wv[kTreeThreads / 32][LG];
    __shared__ int s_wf[kTreeThreads / 32], s_wr[kTreeThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const long long t0 = (long long)t * kTreeTile;
        const int cnt = (int)min((long long)kTreeTile, E - t0);
        // rows that start inside the tile: [ra, rb]; the first kTreeThreads of them are fetched alongside the entries
        const int ra = __ldg(tile_row0 + t), rb = __ldg(tile_row0 + t + 1);
        long long rs0 = -1, rz0 = -1;
        if (ra + tid <= rb) {
            rs0 = __ldg(row_ptr + ra + tid);
            rz0 = __ldg(row_ptr + ra + tid + 1);
        }
        // phase 1
        int2 e[kTreeIT];
#pragma unroll
        for (int q = 0; q < kTreeIT; q++) {
            const int i = q * kTreeThreads + tid;
            e[q] = i < cnt ? __ldg(ent + t0 + i) : make_int2(0, 0);
            s_row[tpad(i)] = -1;
        }
        float x[kTreeIT][LG];
#pragma unroll
        for (int q = 0; q < kTreeIT; q++) {
            const int i = q * kTreeThreads + tid;
            if (LG == 2 && L == 2) {
                const float2 v = i < cnt ? __ldg((const float2 *)in + e[q].x) : make_float2(0.f, 0.f);
                x[q][0] = v.x;
                x[q][LG - 1] = v.y;
            } else {
#pragma unroll
                for (int j = 0; j < LG; j++) x[q][j] = (i < cnt && lb + j < L) ? __ldg(in + (size_t)e[q].x * L + lb + j) : 0.0f;
            }
        }
#pragma unroll
        for (int q = 0; q < kTreeIT; q++) {
            const int i = q * kTreeThreads + tid;
            const float w = __int_as_float(e[q].y);
#pragma unroll
            for (int j = 0; j < LG; j++) s_prod[j][tpad(i)] = i < cnt ? __fmul_rn(w, x[q][j]) : 0.0f;
        }
        __syncthreads();  // s_row is cleared
        if (rz0 > rs0 && rs0 >= t0 && rs0 < t0 + cnt) s_row[tpad((int)(rs0 - t0))] = ra + tid;
        for (int r = ra + kTreeThreads + tid; r <= rb; r += kTreeThreads) {
            const long long s = __ldg(row_ptr + r), z = __ldg(row_ptr + r + 1);
            if (z > s && s >= t0 && s < t0 + cnt) s_row[tpad((int)(s - t0))] = r;
        }
        __syncthreads();
        // phase 2: thread-sequential fold of 8 consecutive entries
        float acc[LG], first[LG];
#pragma unroll
        for (int j = 0; j < LG; j++) acc[j] = first[j] = 0.0f;
        int head_row = -1;       // row of the last row start among my entries
        int first_pos = -1;      // position of my first row start
        // (rows that start AND end among my entries are written at once)
#pragma unroll
        for (int k = 0; k < kTreeIT; k++) {
            const int i = tid * kTreeIT + k;
            const int r = s_row[tpad(i)];
            if (r >= 0) {
                if (head_row < 0) {
                    first_pos = i;
#pragma unroll
                    for (int j = 0; j < LG; j++) first[j] = acc[j];
                } else {
#pragma unroll
                    for (int j = 0; j < LG; j++)
                        if (lb + j < L) val[(size_t)head_row * L + lb + j] = acc[j];
                }
                head_row = r;
#pragma unroll
                for (int j = 0; j < LG; j++) acc[j] = 0.0f;
            }
#pragma unroll
            for (int j = 0; j < LG; j++) acc[j] = __fadd_rn(acc[j], s_prod[j][tpad(i)]);
        }
        const bool has = head_row >= 0;
        if (!has) {
#pragma unroll
            for (int j = 0; j < LG; j++) first[j] = acc[j];
        }
        // segmented inclusive scan over the threads of (has, open sum, row): op (l, r) = r.has ? r : (l.has, l.v + r.v, l.row)
        float v[LG];
#pragma unroll
        for (int j = 0; j < LG; j++) v[j] = acc[j];  // has: sum behind my last row start; else: all my entries
        int f = has ? 1 : 0, rw = head_row;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            float vu[LG];
#pragma unroll
            for (int j = 0; j < LG; j++) vu[j] = __shfl_up_sync(0xffffffffu, v[j], o);
            const int fu = __shfl_up_sync(0xffffffffu, f, o), ru = __shfl_up_sync(0xffffffffu, rw, o);
            if (lane >= o && !f) {
#pragma unroll
                for (int j = 0; j < LG; j++) v[j] = __fadd_rn(vu[j], v[j]);
                f = fu;
                rw = ru;
            }
        }
        // exclusive value inside the warp
        float cv[LG];
#pragma unroll
        for (int j = 0; j < LG; j++) cv[j] = __shfl_up_sync(0xffffffffu, v[j], 1);
        int cf = __shfl_up_sync(0xffffffffu, f, 1), cr = __shfl_up_sync(0xffffffffu, rw, 1);
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < LG; j++) cv[j] = 0.0f;
            cf = 0;
            cr = -1;
        }
        if (lane == 31) {
#pragma unroll
            for (int j = 0; j < LG; j++) s_wv[wid][j] = v[j];
            s_wf[wid] = f;
            s_wr[wid] = rw;
        }
        __syncthreads();
        // carry of the preceding warps, combined in warp order
        float pv[LG];
#pragma unroll
        for (int j = 0; j < LG; j++) pv[j] = 0.0f;
        int pf = 0, pr = -1;
        for (int w = 0; w < wid; w++) {
            if (s_wf[w]) {
#pragma unroll
                for (int j = 0; j < LG; j++) pv[j] = s_wv[w][j];
                pf = 1;
                pr = s_wr[w];
            } else {
#pragma unroll
                for (int j = 0; j < LG; j++) pv[j] = __fadd_rn(pv[j], s_wv[w][j]);
            }
        }
        if (!cf) {  // no row start between the beginning of my warp and me: the carry reaches into the preceding warps
#pragma unroll
            for (int j = 0; j < LG; j++) cv[j] = __fadd_rn(pv[j], cv[j]);
            cf = pf;
            cr = pr;
        }
        // (cf, cv, cr) = what is open in front of my entries: started by row cr inside the tile (cf) or before the tile
        if (has) {
            // the open segment ends at my first row start
            if (cf) {
#pragma unroll
                for (int j = 0; j < LG; j++)
                    if (lb + j < L) val[(size_t)cr * L + lb + j] = __fadd_rn(cv[j], first[j]);
            } else {  // I hold the first row start of the tile: everything in front of it belongs to an earlier tile's row
#pragma unroll
                for (int j = 0; j < LG; j++)
                    if (lb + j < L) tile_part[(size_t)t * L + lb + j] = __fadd_rn(cv[j], first[j]);
                if (lb == 0) tile_info[t].x = first_pos;
            }
        }
        if (tid == kTreeThreads - 1) {  // what is open at the end of the tile
            float ov[LG];
            int orow;
            if (has) {
#pragma unroll
                for (int j = 0; j < LG; j++) ov[j] = acc[j];
                orow = head_row;
            } else {
#pragma unroll
                for (int j = 0; j < LG; j++) ov[j] = __fadd_rn(cv[j], acc[j]);
                orow = cf ? cr : -1;
            }
            if (orow >= 0) {
#pragma unroll
                for (int j = 0; j < LG; j++)
                    if (lb + j < L) val[(size_t)orow * L + lb + j] = ov[j];
            } else {  // no row start in the whole tile
#pragma unroll
                for (int j = 0; j < LG; j++)
                    if (lb + j < L) tile_part[(size_t)t * L + lb + j] = ov[j];
                if (lb == 0) tile_info[t].x = -1;
            }
            if (lb == 0) tile_info[t].y = orow;
        }
        __syncthreads();  // shared arrays are reused by the next tile
    }
}

// rows that span tiles + rows without entries.  One thread per tile / per row.
__global__ void __launch_bounds__(kThreads)
k_splat_carry(const int *__restrict__ row_ptr, const int *__restrict__ vtotal, const int2 *__restrict__ tile_info,
              const float *__restrict__ tile_part, float *__restrict__ val, int n_tiles, int L) {
    const int V = __ldg(vtotal);
    const int gsz = gridDim.x * kThreads, g0 = blockIdx.x * kThreads + threadIdx.x;
    for (int t = g0; t < n_tiles; t += gsz) {
        const int row = __ldg(&tile_info[t].y);
        // the row open at the end of tile t started in tile t iff tile t holds a row start
        if (row < 0 || __ldg(&tile_info[t].x) < 0) continue;
        int t2 = t + 1;
        if (t2 >= n_tiles || __ldg(&tile_info[t2].x) == 0) continue;  // the next tile begins with a row start: complete
        // the leading parts of the following tiles, in tile order; loads run kCarryU tiles ahead of the additions
        constexpr int kCarryU = 8;
        bool open = true;
        for (int u0 = t2; open && u0 < n_tiles; u0 += kCarryU) {
            int fp[kCarryU];
#pragma unroll
            for (int q = 0; q < kCarryU; q++) fp[q] = u0 + q < n_tiles ? __ldg(&tile_info[u0 + q].x) : 0;
            for (int l = 0; l < L; l++) {
                float pt[kCarryU];
#pragma unroll
                for (int q = 0; q < kCarryU; q++) pt[q] = u0 + q < n_tiles ? __ldg(tile_part + (size_t)(u0 + q) * L + l) : 0.0f;
                float acc = val[(size_t)row * L + l];
#pragma unroll
                for (int q = 0; q < kCarryU; q++) {
                    if (fp[q] == 0) break;
                    acc = __fadd_rn(acc, pt[q]);
                    if (fp[q] > 0) break;
                }
                val[(size_t)row * L + l] = acc;
            }
#pragma unroll
            for (int q = 0; q < kCarryU; q++)
                if (fp[q] >= 0) open = false;  // a row start (or the end of the tiles) closes the row
        }
    }
    for (int r = g0; r < V; r += gsz)
        if (__ldg(row_ptr + r + 1) == __ldg(row_ptr + r))
            for (int l = 0; l < L; l++) val[(size_t)r * L + l] = 0.0f;
}

// ---------------------------------------------------------------- blur
// One pass new[v] = old[v] + 0.5*(old[n1(v)] + old[n2(v)])  (permutohedral_cpu.h:663-679) for lattices that do not fit
// one CTA (image-scale V).  HBM stream: per vertex one int2 neighbour pair, the vertex's own labels and the result
// move as 64/128-bit vectors (labels packed per vertex: float2 for L = 2, float4 groups for L % 4 == 0); the two
// neighbour gathers hit L1/L2 because vertex ids follow first-touch (scan) order, so lattice neighbours are close
// in memory.  Each thread keeps kBlurU independent elements in flight (all neighbour pairs and own values are
// requested before the first dependent gather); persistent grid-stride over a device-resident V.
constexpr int kBlurU = 4;

template <typename VT> struct BlurVec;
template <> struct BlurVec<float> {
    static __device__ __forceinline__ float zero() { return 0.f; }
    static __device__ __forceinline__ float comb(float o, float a, float b) { return __fadd_rn(o, __fmul_rn(0.5f, __fadd_rn(a, b))); }
};
template <> struct BlurVec<float2> {
    static __device__ __forceinline__ float2 zero() { return make_float2(0.f, 0.f); }
    static __device__ __forceinline__ float2 comb(float2 o, float2 a, float2 b) {
        return make_float2(BlurVec<float>::comb(o.x, a.x, b.x), BlurVec<float>::comb(o.y, a.y, b.y));
    }
};
template <> struct BlurVec<float4> {
    static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    static __device__ __forceinline__ float4 comb(float4 o, float4 a, float4 b) {
        return make_float4(BlurVec<float>::comb(o.x, a.x, b.x), BlurVec<float>::comb(o.y, a.y, b.y),
                           BlurVec<float>::comb(o.z, a.z, b.z), BlurVec<float>::comb(o.w, a.w, b.w));
    }
};

// G = vectors per vertex (L / lanes of VT); element t = v * G + g
template <typename VT>
__global__ void __launch_bounds__(kThreads)
k_blur_vec(const int2 *__restrict__ nbr_j, const VT *__restrict__ src, VT *__restrict__ dst,
           const int *__restrict__ vtotal, int G) {
    const long long total = (long long)__ldg(vtotal) * G;
    const long long step = (long long)gridDim.x * kThreads * kBlurU;
    for (long long base = (long long)blockIdx.x * kThreads * kBlurU + threadIdx.x; base < total; base += step) {
        int2 nb[kBlurU];
        VT o[kBlurU];
        int g[kBlurU];
#pragma unroll
        for (int u = 0; u < kBlurU; u++) {
            const long long t = base + (long long)u * kThreads;
            nb[u] = make_int2(-1, -1);
            o[u] = BlurVec<VT>::zero();
            g[u] = 0;
            if (t < total) {
                const int v = G == 1 ? (int)t : (int)(t / G);
                g[u] = G == 1 ? 0 : (int)(t - (long long)v * G);
                nb[u] = __ldg(nbr_j + v);
                o[u] = __ldg(src + t);
            }
        }
#pragma unroll
        for (int u = 0; u < kBlurU; u++) {
            const long long t = base + (long long)u * kThreads;
            const VT a = nb[u].x >= 0 ? __ldg(src + (size_t)nb[u].x * G + g[u]) : BlurVec<VT>::zero();
            const VT b = nb[u].y >= 0 ? __ldg(src + (size_t)nb[u].y * G + g[u]) : BlurVec<VT>::zero();
            if (t < total) __stcs(dst + t, BlurVec<VT>::comb(o[u], a, b));
        }
    }
}

// ---- the same pass with its two STREAMS -- the neighbour pairs and the vertices' own values -- brought into shared
// memory by the bulk-copy engine (cp.async.bulk global -> shared, completion on an mbarrier; SASS: UBLKCP) through a ring
// of 2-3 tiles, so that the LSU and the registers only carry the two dependent neighbour gathers and the result.
// Tiles of kBulkTV vertices; one elected thread arms the stage's barrier with the byte count and issues both copies,
// every thread waits on the barrier's phase, consumes, and the block barrier behind the tile frees the stage.
// VT = float2 (L = 2) or float4 (L = 4): one vector per vertex.  The tail (V % kBulkTV) takes plain loads.
// (tile, stages, CTAs per SM) from a sweep on B200 (profiles/r02m_sweeps.txt, scripts/blur_probe.py; 2048 x 2048 stress lattice):
// L = 2: (1024, 3, 3) 0.89-0.90 of the measured HBM peak, plain loads 0.78;  L = 4: (1024, 2, 3) 0.88, plain loads 0.86
constexpr int kBulkTV = 1024, kBulkThreads = 256;
template <typename VT> struct BulkCfg;
template <> struct BulkCfg<float2> { static constexpr int kStages = 3, kPerSm = 3; };
template <> struct BulkCfg<float4> { static constexpr int kStages = 2, kPerSm = 3; };

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

template <typename VT>
__global__ void __launch_bounds__(kBulkThreads)
k_blur_bulk(const int2 *__restrict__ nbr_j, const VT *__restrict__ src, VT *__restrict__ dst, const int *__restrict__ vtotal) {
    constexpr int kBulkStages = BulkCfg<VT>::kStages;
    extern __shared__ __align__(128) unsigned char s_bulk[];
    __shared__ __align__(8) uint64_t s_bar[kBulkStages];
    int2 *s_nb = (int2 *)s_bulk;                                                   // [stages][kBulkTV]
    VT *s_own = (VT *)(s_bulk + (size_t)kBulkStages * kBulkTV * sizeof(int2));     // [stages][kBulkTV]
    const int tid = threadIdx.x;
    const int V = __ldg(vtotal);
    const int n_full = V / kBulkTV;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kBulkStages; s++) mbar_init(&s_bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int k) {  // thread 0: tile k of this CTA into stage k % kBulkStages
        const long long tile = (long long)blockIdx.x + (long long)k * gridDim.x;
        if (tile >= n_full) return;
        const int s = k % kBulkStages;
        mbar_expect_tx(&s_bar[s], (uint32_t)(kBulkTV * (sizeof(int2) + sizeof(VT))));
        bulk_g2s(s_nb + (size_t)s * kBulkTV, nbr_j + tile * kBulkTV, (uint32_t)(kBulkTV * sizeof(int2)), &s_bar[s]);
        bulk_g2s(s_own + (size_t)s * kBulkTV, src + tile * kBulkTV, (uint32_t)(kBulkTV * sizeof(VT)), &s_bar[s]);
    };
    if (tid == 0)
        for (int k = 0; k < kBulkStages; k++) issue(k);
    for (int k = 0;; k++) {
        const long long tile = (long long)blockIdx.x + (long long)k * gridDim.x;
        if (tile >= n_full) break;
        const int s = k % kBulkStages;
        mbar_wait(&s_bar[s], (uint32_t)((k / kBulkStages) & 1));
        constexpr int U = kBulkTV / kBulkThreads;
        int2 nb[U];
        VT o[U], a[U], b[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            nb[u] = s_nb[(size_t)s * kBulkTV + u * kBulkThreads + tid];
            o[u] = s_own[(size_t)s * kBulkTV + u * kBulkThreads + tid];
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            a[u] = nb[u].x >= 0 ? __ldg(src + nb[u].x) : BlurVec<VT>::zero();
            b[u] = nb[u].y >= 0 ? __ldg(src + nb[u].y) : BlurVec<VT>::zero();
        }
#pragma unroll
        for (int u = 0; u < U; u++) __stcs(dst + tile * kBulkTV + u * kBulkThreads + tid, BlurVec<VT>::comb(o[u], a[u], b[u]));
        __syncthreads();  // stage s is consumed
        if (tid == 0) issue(k + kBulkStages);
    }
    // tail
    for (long long t = (long long)n_full * kBulkTV + (long long)blockIdx.x * kBulkThreads + tid; t < V; t += (long long)gridDim.x * kBulkThreads) {
        const int2 nbv = __ldg(nbr_j + t);
        const VT ov = __ldg(src + t);
        const VT av = nbv.x >= 0 ? __ldg(src + nbv.x) : BlurVec<VT>::zero();
        const VT bv = nbv.y >= 0 ? __ldg(src + nbv.y) : BlurVec<VT>::zero();
        __stcs(dst + t, BlurVec<VT>::comb(ov, av, bv));
    }
}

// all D blur passes of one problem inside one CTA: replaces D launch-bound passes when a batch holds several
// problems or the lattice is small.  When values (ping-pong) AND the problem's D neighbour tables fit shared memory
// everything is fetched in one round of independent global loads and the passes run from shared memory; otherwise
// the values ping-pong in shared memory with neighbour pairs read per pass, or (huge lattices) in global memory.
constexpr int kBlurFusedBytes = 160 * 1024;
__global__ void __launch_bounds__(1024)
k_blur_fused(const int2 *__restrict__ nbr, int Vcap, const int *__restrict__ vbase, float *__restrict__ A,
             float *__restrict__ B, int L, int D) {
    extern __shared__ float s_blur[];
    const int b = blockIdx.x;
    const int vb = __ldg(vbase + b);
    const int nv = __ldg(vbase + b + 1) - vb;
    const int n = nv * L;
    float *gA = A + (size_t)vb * L, *gB = B + (size_t)vb * L;
    if ((size_t)2 * n * sizeof(float) + (size_t)D * nv * sizeof(int2) <= (size_t)kBlurFusedBytes) {
        float *src = s_blur, *dst = s_blur + n;
        int2 *s_nb = (int2 *)(s_blur + 2 * n + ((2 * n) & 1));  // 8-byte aligned
        for (int t = threadIdx.x; t < n; t += 1024) src[t] = gA[t];
        for (int t = threadIdx.x; t < D * nv; t += 1024) {
            const int j = t / nv, v = t - j * nv;
            s_nb[t] = __ldg(nbr + (size_t)j * Vcap + vb + v);
        }
        __syncthreads();
        for (int j = 0; j < D; j++) {
            for (int t = threadIdx.x; t < n; t += 1024) {
                const int v = t / L, l = t - v * L;
                const int2 nb = s_nb[j * nv + v];
                const float a = nb.x >= 0 ? src[(nb.x - vb) * L + l] : 0.f;
                const float c = nb.y >= 0 ? src[(nb.y - vb) * L + l] : 0.f;
                dst[t] = __fadd_rn(src[t], __fmul_rn(0.5f, __fadd_rn(a, c)));
            }
            __syncthreads();
            float *tmp = src;
            src = dst;
            dst = tmp;
        }
        for (int t = threadIdx.x; t < n; t += 1024) gB[t] = src[t];
    } else if ((size_t)2 * n * sizeof(float) <= (size_t)kBlurFusedBytes) {
        float *src = s_blur, *dst = s_blur + n;
        for (int t = threadIdx.x; t < n; t += 1024) src[t] = gA[t];
        __syncthreads();
        for (int j = 0; j < D; j++) {
            const int2 *nb_j = nbr + (size_t)j * Vcap + vb;
            for (int t = threadIdx.x; t < n; t += 1024) {
                const int v = t / L, l = t - v * L;
                const int2 nb = __ldg(nb_j + v);
                const float a = nb.x >= 0 ? src[(nb.x - vb) * L + l] : 0.f;
                const float c = nb.y >= 0 ? src[(nb.y - vb) * L + l] : 0.f;
                dst[t] = __fadd_rn(src[t], __fmul_rn(0.5f, __fadd_rn(a, c)));
            }
            __syncthreads();
            float *tmp = src;
            src = dst;
            dst = tmp;
        }
        for (int t = threadIdx.x; t < n; t += 1024) gB[t] = src[t];
    } else {
        float *src = gA, *dst = gB;
        for (int j = 0; j < D; j++) {
            const int2 *nb_j = nbr + (size_t)j * Vcap + vb;
            for (int t = threadIdx.x; t < n; t += 1024) {
                const int v = t / L, l = t - v * L;
                const int2 nb = __ldg(nb_j + v);
                const float a = nb.x >= 0 ? src[(size_t)(nb.x - vb) * L + l] : 0.f;
                const float c = nb.y >= 0 ? src[(size_t)(nb.y - vb) * L + l] : 0.f;
                dst[t] = __fadd_rn(src[t], __fmul_rn(0.5f, __fadd_rn(a, c)));
            }
            __syncthreads();
            float *tmp = src;
            src = dst;
            dst = tmp;
        }
        if (src != gB)
            for (int t = threadIdx.x; t < n; t += 1024) gB[t] = src[t];
    }
}

// ---------------------------------------------------------------- slice (+ fused Potts apply)
enum SliceMode { kPlain = 0, kApplyFirst = 1, kApplyAdd = 2 };

template <int MODE>
__global__ void __launch_bounds__(kThreads)
k_slice(const int *__restrict__ offset, const float *__restrict__ bary, const float *__restrict__ val,
        float *__restrict__ out, int NT, int D, int L, float alpha, float w, const float *__restrict__ norm,
        const float *__restrict__ unary) {
    const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (t >= (long long)NT * L) return;
    const int i = (int)(t / L), l = (int)(t - (long long)i * L);
    float s = 0.0f;
    for (int r = 0; r < D; r++) {
        const int id = __ldg(offset + (size_t)i * D + r);
        const float wa = __fmul_rn(__ldg(bary + (size_t)i * D + r), alpha);
        s = __fadd_rn(s, __fmul_rn(wa, __ldg(val + (size_t)id * L + l)));
    }
    if (MODE == kPlain) {
        out[t] = s;
    } else {
        const float m = __fmul_rn(__fmul_rn(w, __ldg(norm + i)), s);  // (w_*norm_[i])*tmp[k]
        const float base = MODE == kApplyFirst ? -__ldg(unary + t) : out[t];
        out[t] = __fadd_rn(base, m);
    }
}

__global__ void k_norm_finish(float *__restrict__ norm, int NT) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i < NT) norm[i] = __fdiv_rn(1.0f, __fadd_rn(norm[i], 1e-20f));  // pairwise3d.h:26
}

__global__ void k_fill(float *__restrict__ x, float v, int n) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i < n) x[i] = v;
}

}  // namespace

// splat + all blur passes; *values_out is the buffer holding the blurred vertex values
int filter_splat_blur(Ctx *ctx, const Batch &b, LatticeSet *ls, const float *in_dev, int L, const float **values_out) {
    cudaStream_t st = ctx->stream;
    if (L > ls->Lmax) return fail(LCCRF_ERR_ARG, "filter: L exceeds the lattice workspace");
    const int D = ls->D;
    const int *vt = ls->vbase + ls->B;
    float *src = ls->valA, *dst = ls->valB;
    const bool split = b.NT > 0 && ctx->opt_ordered_splat && ctx->opt_split_splat && ls->max_chunks > 0 &&
                       ctx_concurrent(ctx) && ctx->sub_stream[ctx->branch];
    if (b.NT > 0 && !ctx->opt_ordered_splat) {
        // tree splat: one streaming pass over the sorted entries per label group + the cross-tile carries
        const long long E = (long long)b.NT * D;
        const int grid = ls->n_tiles < kNumSMs * 8 ? ls->n_tiles : kNumSMs * 8;
        const int LG = L == 1 ? 1 : (L == 2 ? 2 : 4);
        for (int lb = 0; lb < L; lb += LG) {
            LCCRF_KERNEL(ctx, "k_splat_tree");
            if (LG == 1) k_splat_tree<1><<<grid, kTreeThreads, 0, st>>>(ls->row_ptr, ls->tile_row0, ls->csr_ent, in_dev, src, ls->tile_part, ls->tile_info, ls->n_tiles, E, L, lb);
            else if (LG == 2) k_splat_tree<2><<<grid, kTreeThreads, 0, st>>>(ls->row_ptr, ls->tile_row0, ls->csr_ent, in_dev, src, ls->tile_part, ls->tile_info, ls->n_tiles, E, L, lb);
            else k_splat_tree<4><<<grid, kTreeThreads, 0, st>>>(ls->row_ptr, ls->tile_row0, ls->csr_ent, in_dev, src, ls->tile_part, ls->tile_info, ls->n_tiles, E, L, lb);
        }
        {
            LCCRF_KERNEL(ctx, "k_splat_carry");
            const int cg = persistent_grid(ls->n_tiles > ls->Vcap ? ls->n_tiles : ls->Vcap, kThreads, 4);
            k_splat_carry<<<cg, kThreads, 0, st>>>(ls->row_ptr, vt, ls->tile_info, ls->tile_part, src, ls->n_tiles, L);
        }
    } else if (b.NT > 0) {
        const long long E = (long long)b.NT * D;
        const int LG = tile_labels(L);
        const int grid = ls->n_tiles < kNumSMs * 12 ? ls->n_tiles : kNumSMs * 12;
        const size_t smem = (size_t)kRowsWin * LG * sizeof(float);
        LCCRF_TRY(ensure_dyn_smem(ctx, k_splat_rows<4>, (int)((size_t)kRowsWin * 4 * sizeof(float))));
        // the short rows and the long rows of a lattice are disjoint sets of vertex rows: the short-row kernel (bound by
        // L2 gathers) runs beside the long-row scan kernels (bound by instruction issue) on the branch's sub-stream
        cudaStream_t rs = st;
        if (split) {
            rs = ctx->sub_stream[ctx->branch];
            LCCRF_CUDA(cudaEventRecord(ctx->ev_sub_fork[ctx->branch], st));
            LCCRF_CUDA(cudaStreamWaitEvent(rs, ctx->ev_sub_fork[ctx->branch], 0));
        }
        for (int lb = 0; lb < L; lb += LG) {
            LCCRF_KERNEL(ctx, "k_splat_rows");
            switch (LG) {
                case 1: k_splat_rows<1><<<grid, kRowsThreads, smem, rs>>>(ls->row_ptr, ls->tile_row0, ls->tile_own, ls->csr_ent, in_dev, src, ls->n_tiles, E, L, lb); break;
                case 2: k_splat_rows<2><<<grid, kRowsThreads, smem, rs>>>(ls->row_ptr, ls->tile_row0, ls->tile_own, ls->csr_ent, in_dev, src, ls->n_tiles, E, L, lb); break;
                default: k_splat_rows<4><<<grid, kRowsThreads, smem, rs>>>(ls->row_ptr, ls->tile_row0, ls->tile_own, ls->csr_ent, in_dev, src, ls->n_tiles, E, L, lb); break;
            }
        }
    }
    // long rows (>= kLongRow entries): speculative parallel scan.  The lists live on the device, so the grids are
    // sized for the worst case a lattice set can hold and capped at a few waves (grid-stride inside).
    if (b.NT > 0 && ls->max_chunks > 0 && ctx->opt_ordered_splat) {
        const long long maxc = (long long)ls->max_chunks * ((L + 1) / 2), maxr = (long long)ls->max_long * L;
        const int gk = (int)(maxc < kNumSMs * 3 ? maxc : kNumSMs * 3);  // compose: persistent, one resident wave
        const int gr = (int)(maxr < kNumSMs * 8 ? maxr : kNumSMs * 8);
        const int4 *desc = (const int4 *)ls->chunk_desc;
        {
            LCCRF_KERNEL(ctx, "k_scan_compose");
            if (scan_labels(L) == 1) k_scan_compose<1><<<gk, 256, 0, st>>>(ls->row_ptr, ls->csr_ent, in_dev, ls->row_list_long, ls->row_counts, ls->long_chunk0, desc, ls->chunk_sum, (ChunkRec *)ls->chunk_rec, L);
            else k_scan_compose<2><<<gk, 256, 0, st>>>(ls->row_ptr, ls->csr_ent, in_dev, ls->row_list_long, ls->row_counts, ls->long_chunk0, desc, ls->chunk_sum, (ChunkRec *)ls->chunk_rec, L);
        }
        { LCCRF_KERNEL(ctx, "k_scan_walk");
          k_scan_walk<<<gr, 256, 0, st>>>(ls->row_ptr, ls->csr_ent, in_dev, src, ls->row_list_long, ls->row_counts, ls->long_chunk0, (const ChunkRec *)ls->chunk_rec, ls->chunk_sum, L); }
    }
    if (split) {
        LCCRF_CUDA(cudaEventRecord(ctx->ev_sub_join[ctx->branch], ctx->sub_stream[ctx->branch]));
        LCCRF_CUDA(cudaStreamWaitEvent(st, ctx->ev_sub_join[ctx->branch], 0));
    }
    if (b.fused_blur) {  // one CTA per problem runs all D passes
        LCCRF_TRY(ensure_dyn_smem(ctx, k_blur_fused, kBlurFusedBytes + 16));
        LCCRF_KERNEL(ctx, "k_blur_fused");
        k_blur_fused<<<b.B, 1024, kBlurFusedBytes + 16, st>>>(ls->nbr, ls->Vcap, ls->vbase, src, dst, L, D);
        *values_out = dst;
        LCCRF_CUDA(cudaGetLastError());
        return LCCRF_OK;
    }
    // vector width: the widest of float4 / float2 / float that divides L (value rows are L floats, 16-byte aligned
    // bases, so vertex v's row is aligned to the vector whenever the width divides L)
    const int W = (L % 4 == 0) ? 4 : (L % 2 == 0) ? 2 : 1;
    const int G = L / W;
    const int bgrid = persistent_grid(((long long)ls->Vcap * G + kBlurU - 1) / kBlurU, kThreads, 8);
    for (int j = 0; j < D; j++) {
        const int2 *nb = ls->nbr + (size_t)j * ls->Vcap;
        const bool bulk = ctx->opt_bulk_blur && G == 1 && (W == 2 || W == 4) && (((size_t)nb & 15) == 0);
        if (bulk) {
            // streams through the bulk-copy engine (UBLKCP); 16-byte aligned neighbour tables (Vcap is even)
            const int stages = W == 2 ? BulkCfg<float2>::kStages : BulkCfg<float4>::kStages;
            const int per_sm = W == 2 ? BulkCfg<float2>::kPerSm : BulkCfg<float4>::kPerSm;
            const size_t smem = (size_t)stages * kBulkTV * (sizeof(int2) + (W == 2 ? sizeof(float2) : sizeof(float4)));
            const long long tiles = (long long)ls->Vcap / kBulkTV + 1;
            const int grid = (int)(tiles < (long long)kNumSMs * per_sm ? tiles : (long long)kNumSMs * per_sm);
            LCCRF_KERNEL(ctx, "k_blur");
            if (W == 2) {
                LCCRF_TRY(ensure_dyn_smem(ctx, k_blur_bulk<float2>, (int)smem));
                k_blur_bulk<float2><<<grid, kBulkThreads, smem, st>>>(nb, (const float2 *)src, (float2 *)dst, vt);
            } else {
                LCCRF_TRY(ensure_dyn_smem(ctx, k_blur_bulk<float4>, (int)smem));
                k_blur_bulk<float4><<<grid, kBulkThreads, smem, st>>>(nb, (const float4 *)src, (float4 *)dst, vt);
            }
        } else {
            LCCRF_KERNEL(ctx, "k_blur");
            if (W == 4) k_blur_vec<float4><<<bgrid, kThreads, 0, st>>>(nb, (const float4 *)src, (float4 *)dst, vt, G);
            else if (W == 2) k_blur_vec<float2><<<bgrid, kThreads, 0, st>>>(nb, (const float2 *)src, (float2 *)dst, vt, G);
            else k_blur_vec<float><<<bgrid, kThreads, 0, st>>>(nb, src, dst, vt, G);
        }
        float *t = src;
        src = dst;
        dst = t;
    }
    *values_out = src;
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

static int launch_slice(Ctx *ctx, int mode, const Batch &b, LatticeSet *ls, const float *values, float *out,
                        int L, const float *unary) {
    if (b.NT == 0) return LCCRF_OK;
    const int grid = cdiv((long long)b.NT * L, kThreads);
    cudaStream_t st = ctx->stream;
    LCCRF_KERNEL(ctx, "k_slice");
    if (mode == kPlain)
        k_slice<kPlain><<<grid, kThreads, 0, st>>>(ls->offset, ls->bary, values, out, b.NT, ls->D, L, ls->alpha, 0.f, nullptr, nullptr);
    else if (mode == kApplyFirst)
        k_slice<kApplyFirst><<<grid, kThreads, 0, st>>>(ls->offset, ls->bary, values, out, b.NT, ls->D, L, ls->alpha, ls->w, ls->norm, unary);
    else
        k_slice<kApplyAdd><<<grid, kThreads, 0, st>>>(ls->offset, ls->bary, values, out, b.NT, ls->D, L, ls->alpha, ls->w, ls->norm, nullptr);
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

// PermutohedralLatticeCPU::compute(out, in, L)
int filter_full(Ctx *ctx, const Batch &b, LatticeSet *ls, float *out_dev, const float *in_dev, int L) {
    const float *vals = nullptr;
    LCCRF_TRY(filter_splat_blur(ctx, b, ls, in_dev, L, &vals));
    return launch_slice(ctx, kPlain, b, ls, vals, out_dev, L, nullptr);
}

// PottsPotential3D ctor: norm_ = 1/(filter(1)+1e-20)   pairwise3d.h:22-27
int potts_norm(Ctx *ctx, const Batch &b, LatticeSet *ls) {
    if (b.NT == 0) return LCCRF_OK;
    { LCCRF_KERNEL(ctx, "k_fill"); k_fill<<<cdiv(b.NT, kThreads), kThreads, 0, ctx->stream>>>(ls->norm, 1.0f, b.NT); }
    const float *vals = nullptr;
    LCCRF_TRY(filter_splat_blur(ctx, b, ls, ls->norm, 1, &vals));
    LCCRF_TRY(launch_slice(ctx, kPlain, b, ls, vals, ls->norm, 1, nullptr));
    { LCCRF_KERNEL(ctx, "k_norm_finish"); k_norm_finish<<<cdiv(b.NT, kThreads), kThreads, 0, ctx->stream>>>(ls->norm, b.NT); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

// PottsPotential3D::apply on arbitrary device arrays: tmp = filter(in); out += (w*norm)*tmp
int mf_potts_apply(Ctx *ctx, const Batch &b, LatticeSet *ls, float *out, const float *in, float *tmp, int L) {
    LCCRF_TRY(filter_full(ctx, b, ls, tmp, in, L));
    if (b.NT > 0) LCCRF_TRY(launch_axpy_norm(ctx, out, tmp, ls->norm, ls->w, b.NT, L));
    return LCCRF_OK;
}

// one potential of a mean-field step: next = (first ? -unary : next) + (w*norm)*filter(cur)
int mf_apply_fused(Ctx *ctx, const Batch &b, LatticeSet *ls, const float *cur, float *next, const float *unary,
                   bool first) {
    const float *vals = nullptr;
    LCCRF_TRY(filter_splat_blur(ctx, b, ls, cur, b.L, &vals));
    return launch_slice(ctx, first ? kApplyFirst : kApplyAdd, b, ls, vals, next, b.L, unary);
}

}  // namespace lccrf
