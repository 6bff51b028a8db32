// unary_obs_check.cu -- device checks of the straight-line arithmetic of k_map_point_unary (csrc/unary_obs.cuh)
// against the library sequences it stands in for.  Built with the library's nvcc flags and run by
// tests/test_gpu_unary_obs.py; prints one summary line of counters ("unary_obs k=v ...") and exits 0 when the
// program ran (the test judges the counters).
//   rcp   every float bit pattern: rcp_fast == __frcp_rn wherever rcp_undecided is false, and rcp_undecided is true
//         exactly for the exponent fields outside [1, 252]
//   bnd   s placed so that sqrt(s) sits at every offset in +-2^15 double ulps of a float rounding midpoint (exact
//         midpoints included), for floats across the binades of s in [2^-60, 2^60]: (float)sqrt_newton(s) ==
//         (float)__dsqrt_rn(s) wherever the fast path decides; largest |sqrt_newton(s) - __dsqrt_rn(s)| in double ulps
//   rnd   log-uniform random s in [2^-60, 2^60): the same check, and the rate at which the fast path gives up
//   spc   the limits of the range check (2^-60, 2^60, their neighbours), 0, subnormal doubles, Inf and NaN
//   e2e   observe_fast against observe on random and crafted (pose, point, camera, keypoint) tuples: whenever
//         observe_fast does not flag, er and dz are bit-identical
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include <cuda_runtime.h>

#include "unary_obs.cuh"

using namespace lccrf;

enum {
    RCP_N, RCP_BAD, RCP_FLAG_BAD, RCP_FLAGGED,
    BND_N, BND_BAD, BND_FLAGGED, BND_MARGIN,
    RND_N, RND_BAD, RND_FLAGGED, RND_MARGIN,
    SPC_N, SPC_BAD,
    E2E_N, E2E_BAD, E2E_FLAGGED, E2E_KEPT, E2E_NAN,
    FIRST_BAD_E2E,
    NCNT
};
static const char *kNames[NCNT] = {
    "rcp_n", "rcp_bad", "rcp_flag_bad", "rcp_flagged",
    "bnd_n", "bnd_bad", "bnd_flagged", "bnd_margin_ulps",
    "rnd_n", "rnd_bad", "rnd_flagged", "rnd_margin_ulps",
    "spc_n", "spc_bad",
    "e2e_n", "e2e_bad", "e2e_flagged", "e2e_kept", "e2e_nan",
    "first_bad_e2e",
};

#define CK(x)                                                                                   \
    do {                                                                                        \
        cudaError_t e_ = (x);                                                                   \
        if (e_ != cudaSuccess) {                                                                \
            fprintf(stderr, "%s:%d: %s\n", __FILE__, __LINE__, cudaGetErrorString(e_));         \
            exit(2);                                                                            \
        }                                                                                       \
    } while (0)

constexpr int kThreads = 256;

__device__ __forceinline__ uint64_t splitmix(uint64_t x) {
    x += 0x9e3779b97f4a7c15ull;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

struct Rng {
    uint64_t s;
    __device__ uint64_t next() { return s = splitmix(s); }
    __device__ unsigned u32(unsigned n) { return (unsigned)((next() >> 32) % n); }
    __device__ float uni(float a, float b) { return a + (b - a) * (float)(next() >> 40) * 0x1p-24f; }
};

// the fast path's verdict on a square root: sqrt_newton's value is used unless s is outside (2^-60, 2^60) or the value
// lies near a float rounding midpoint (the two tests of observe_fast)
__device__ __forceinline__ bool sqrt_flag(double s, double y) { return !(s > 0x1p-60 && s < 0x1p60) || sqrt_near_midpoint(y); }

__device__ __forceinline__ unsigned long long ulp_dist(double a, double b) {
    const long long d = __double_as_longlong(a) - __double_as_longlong(b);
    return (unsigned long long)(d < 0 ? -d : d);
}

// one square root: counters [n, bad, flagged, margin] at c
__device__ __forceinline__ void check_sqrt(double s, unsigned long long (&c)[4]) {
    const double y = sqrt_newton(s), r = __dsqrt_rn(s);
    const bool f = sqrt_flag(s, y);
    c[0]++;
    c[2] += f;
    if (!f && __float_as_uint((float)y) != __float_as_uint((float)r)) c[1]++;
    const unsigned long long m = ulp_dist(y, r);
    if (m > c[3]) c[3] = m;
}

__device__ void flush(unsigned long long *cnt, int base, const unsigned long long (&c)[4], bool margin) {
    atomicAdd(cnt + base, c[0]);
    atomicAdd(cnt + base + 1, c[1]);
    atomicAdd(cnt + base + 2, c[2]);
    if (margin) atomicMax(cnt + base + 3, c[3]);
    else atomicAdd(cnt + base + 3, c[3]);
}

__global__ void k_rcp(unsigned long long *cnt) {
    unsigned long long c[4] = {0, 0, 0, 0};  // n, bad, flag_bad, flagged
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < (1ull << 32); i += (uint64_t)gridDim.x * blockDim.x) {
        const float z = __uint_as_float((unsigned)i);
        const float r = rcp_fast(z);
        const bool f = rcp_undecided(z);
        const unsigned e = ((unsigned)i >> 23) & 255u;
        c[0]++;
        c[2] += f != (e < 1 || e > 252);
        c[3] += f;
        if (!f && __float_as_uint(r) != __float_as_uint(__frcp_rn(z))) c[1]++;
    }
    atomicAdd(cnt + RCP_N, c[0]);
    atomicAdd(cnt + RCP_BAD, c[1]);
    atomicAdd(cnt + RCP_FLAG_BAD, c[2]);
    atomicAdd(cnt + RCP_FLAGGED, c[3]);
}

constexpr int kBndE0 = -30, kBndE1 = 30;  // binades [2^E, 2^(E+1)) of sqrt(s): s in [2^-60, 2^60)
constexpr int kBndPerBinade = 64;          // floats per binade: the 2 lowest and 2 highest mantissas + 60 random
constexpr int kBndHalf = 1 << 15;          // offsets -2^15 .. 2^15 double ulps around the midpoint

__global__ void k_bnd(unsigned long long *cnt) {
    unsigned long long c[4] = {0, 0, 0, 0};
    const uint64_t per_f = 2 * kBndHalf + 1, nf = (uint64_t)(kBndE1 - kBndE0) * kBndPerBinade;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < nf * per_f; i += (uint64_t)gridDim.x * blockDim.x) {
        const int fi = (int)(i / per_f), k = (int)(i % per_f) - kBndHalf;
        const int E = kBndE0 + fi / kBndPerBinade, j = fi % kBndPerBinade;
        const unsigned mant = j == 0 ? 0u : j == 1 ? 1u : j == 2 ? 0x7fffffu : j == 3 ? 0x7ffffeu
                                                                 : (unsigned)(splitmix(fi) >> 41);
        // f = (1 + mant 2^-23) 2^E; its upper rounding midpoint m = f + 2^(E-24) (25 bits: exact); t = m + k 2^(E-52)
        const double m = ldexp(1.0 + mant * 0x1p-23 + 0x1p-24, E);
        const double t = __dadd_rn(m, ldexp((double)k, E - 52));
        check_sqrt(__dmul_rn(t, t), c);  // k = 0: s = m^2 exactly, sqrt(s) is the midpoint itself
    }
    flush(cnt, BND_N, c, true);
}

__global__ void k_rnd(unsigned long long *cnt, uint64_t n, uint64_t seed) {
    unsigned long long c[4] = {0, 0, 0, 0};
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t h = splitmix(i ^ seed), h2 = splitmix(h);
        const int e = -60 + (int)(h2 % 120);
        const double s = __hiloint2double((int)(((unsigned)(1023 + e) << 20) | (unsigned)((h >> 32) & 0xfffffu)), (int)(unsigned)h);
        check_sqrt(s, c);
    }
    flush(cnt, RND_N, c, true);
}

__global__ void k_spc(unsigned long long *cnt) {
    if (blockIdx.x || threadIdx.x) return;
    const double lo = 0x1p-60, hi = 0x1p60, inf = __longlong_as_double(0x7ff0000000000000ll);
    // must be flagged: at or outside the limits, 0, subnormal, Inf, NaN
    const double out[] = {lo, nextafter(lo, 0.0), 0.5 * lo, hi, nextafter(hi, inf), 2.0 * hi, 0.0, -0.0,
                          __longlong_as_double(1ll), __longlong_as_double(0x000fffffffffffffll), 0x1p-1022, 0x1p-700,
                          0x1p700, 0x1.fffffffffffffp1023, inf, __longlong_as_double(0x7ff8000000000000ll),
                          __longlong_as_double(0xfff8000000000000ll), -1.0};
    // just inside: decided correctly or flagged
    const double in[] = {nextafter(lo, inf), nextafter(nextafter(lo, inf), inf), nextafter(hi, 0.0), 1.0};
    for (double s : out) {
        const double y = sqrt_newton(s);
        cnt[SPC_N]++;
        if (!sqrt_flag(s, y)) {
            cnt[SPC_BAD]++;
            printf("spc: s = %a not flagged\n", s);
        }
    }
    for (double s : in) {
        const double y = sqrt_newton(s);
        cnt[SPC_N]++;
        if (!sqrt_flag(s, y) && __float_as_uint((float)y) != __float_as_uint((float)__dsqrt_rn(s))) {
            cnt[SPC_BAD]++;
            printf("spc: s = %a decided wrongly\n", s);
        }
    }
}

// z values at the reciprocal's edges: exponent fields 0, 1, 2, 126, 127, 252, 253, 254 (random mantissa), +-0, +-Inf,
// NaN, the extremes of the subnormals and normals; either sign
__device__ float edge_z(Rng &r) {
    const unsigned fields[8] = {0, 1, 2, 126, 127, 252, 253, 254};
    const unsigned sign = (r.u32(4) == 0) << 31;
    const unsigned pick = r.u32(16);
    unsigned b;
    if (pick < 8) b = (fields[pick] << 23) | (unsigned)(r.next() >> 41);
    else if (pick == 8) b = 0;
    else if (pick == 9) b = 0x7f800000u;
    else if (pick == 10) b = 0x7fc00000u;
    else if (pick == 11) b = 1;
    else if (pick == 12) b = 0x007fffffu;
    else if (pick == 13) b = 0x00800000u;
    else if (pick == 14) b = 0x7f7fffffu;
    else b = 0x7e800000u - (unsigned)r.u32(3);  // the top of field 252 and its neighbours
    return __uint_as_float(b | sign);
}

// residual components for the crafted-residual tuples (u = a, v = b, keypoint (0, 0): s = a^2 + b^2 exactly)
__device__ float edge_res(Rng &r) {
    switch (r.u32(12)) {
    case 0: return 0.f;
    case 1: return 0x1p-30f;                       // s = 2^-60: flagged
    case 2: return 0x1.000002p-30f;                // just above 2^-60
    case 3: return 0x1.fffffep-31f;                // just below 2^-60
    case 4: return 0x1p30f;                        // s = 2^60: flagged
    case 5: return 0x1.fffffep29f;                 // just below 2^60
    case 6: return 0x1.000002p30f;                 // just above 2^60
    case 7: return 0x1p-56f;                       // a small second component
    case 8: return __uint_as_float(1u);            // the smallest subnormal
    case 9: return 0x1.fffffep127f;                // FLT_MAX: s ~ 2^256
    default: return ldexpf(r.uni(1.f, 2.f), (int)r.u32(100) - 50) * (r.u32(2) ? 1.f : -1.f);
    }
}

__global__ void k_e2e(unsigned long long *cnt, uint64_t n, uint64_t seed) {
    unsigned long long nn = 0, bad = 0, flagged = 0, kept = 0, nan = 0;
    const float inf = __uint_as_float(0x7f800000u);
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        Rng r{splitmix(i ^ seed)};
        float4 p[3];
        for (int q = 0; q < 3; q++) p[q] = make_float4(r.uni(-1.f, 1.f), r.uni(-1.f, 1.f), r.uni(-1.f, 1.f), r.uni(-3.f, 3.f));
        float x0 = r.uni(-5.f, 5.f), x1 = r.uni(-5.f, 5.f), x2 = r.uni(-1.f, 10.f);
        float4 intr = make_float4(r.uni(200.f, 800.f), r.uni(200.f, 800.f), r.uni(0.f, 640.f), r.uni(0.f, 480.f));
        float4 bnd = make_float4(0.f, 640.f, 0.f, 480.f);
        float2 uv = make_float2(r.uni(0.f, 640.f), r.uni(0.f, 480.f));
        const unsigned cls = r.u32(8);
        if (cls == 0) {  // z at the reciprocal's edges
            p[2] = make_float4(0.f, 0.f, 0.f, edge_z(r));
            if (r.u32(2)) bnd = make_float4(-inf, inf, -inf, inf);
        } else if (cls == 1 || cls == 2) {  // crafted residual: identity pose, unit camera, s = a^2 + b^2
            p[0] = make_float4(1.f, 0.f, 0.f, 0.f);
            p[1] = make_float4(0.f, 1.f, 0.f, 0.f);
            p[2] = make_float4(0.f, 0.f, 1.f, 0.f);
            x0 = edge_res(r);
            x1 = cls == 1 ? 0.f : edge_res(r);
            x2 = 1.f;
            intr = make_float4(1.f, 1.f, 0.f, 0.f);
            bnd = make_float4(-inf, inf, -inf, inf);
            uv = make_float2(0.f, 0.f);
        } else if (cls == 3) {  // 0 * Inf: x = 0 at z = +0 (invz = Inf), or fx * x = Inf at z = Inf (invz = 0)
            p[0] = make_float4(1.f, 0.f, 0.f, 0.f);
            p[1] = make_float4(0.f, 1.f, 0.f, 0.f);
            if (r.u32(2)) {
                p[2] = make_float4(0.f, 0.f, 0.f, 0.f);
                x0 = 0.f;
            } else {
                p[2] = make_float4(0.f, 0.f, 0.f, inf);
                intr.x = 0x1.fffffep127f;
                x0 = 4.f;
            }
            bnd = make_float4(-inf, inf, -inf, inf);
        } else if (cls == 4 || cls == 5) {  // a bound on u or v exactly, or one float ulp either side
            const float xc = row_dot(p[0], x0, x1, x2), yc = row_dot(p[1], x0, x1, x2), zc = row_dot(p[2], x0, x1, x2);
            const float invz = __frcp_rn(zc);
            const float u = __fadd_rn(__fmul_rn(__fmul_rn(intr.x, xc), invz), intr.z);
            const float v = __fadd_rn(__fmul_rn(__fmul_rn(intr.y, yc), invz), intr.w);
            bnd = make_float4(-inf, inf, -inf, inf);
            const float w = (cls == 4) ? u : v;
            const unsigned side = r.u32(3);
            const float b = side == 0 ? w : side == 1 ? nextafterf(w, -inf) : nextafterf(w, inf);
            const unsigned which = r.u32(2);
            if (cls == 4) (which ? bnd.y : bnd.x) = b;
            else (which ? bnd.w : bnd.z) = b;
        } else if (cls == 6) {
            bnd = make_float4(-inf, inf, -inf, inf);  // nothing out of bounds: mostly kept
        }
        const float xc = row_dot(p[0], x0, x1, x2), yc = row_dot(p[1], x0, x1, x2), zc = row_dot(p[2], x0, x1, x2);
        float er, dz, er2, dz2;
        const bool f = observe_fast(xc, yc, zc, intr, bnd, uv, er, dz);
        observe(p[0], p[1], p[2], intr, bnd, x0, x1, x2, uv, er2, dz2);
        nn++;
        flagged += f;
        kept += er2 != 0.f || dz2 != 0.f;
        nan += er2 != er2;
        if (!f) {
            const bool same_e = __float_as_uint(er) == __float_as_uint(er2) || (er != er && er2 != er2);
            const bool same_d = __float_as_uint(dz) == __float_as_uint(dz2) || (dz != dz && dz2 != dz2);
            if (!same_e || !same_d) {
                bad++;
                atomicMin(cnt + FIRST_BAD_E2E, (unsigned long long)i);
            }
        }
    }
    atomicAdd(cnt + E2E_N, nn);
    atomicAdd(cnt + E2E_BAD, bad);
    atomicAdd(cnt + E2E_FLAGGED, flagged);
    atomicAdd(cnt + E2E_KEPT, kept);
    atomicAdd(cnt + E2E_NAN, nan);
}

int main(int argc, char **argv) {
    const uint64_t n_rnd = argc > 1 ? strtoull(argv[1], nullptr, 0) : (1ull << 30);
    const uint64_t n_e2e = argc > 2 ? strtoull(argv[2], nullptr, 0) : (1ull << 28);
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    unsigned long long h[NCNT] = {0}, *d = nullptr;
    h[FIRST_BAD_E2E] = ~0ull;
    CK(cudaMalloc(&d, sizeof(h)));
    CK(cudaMemcpy(d, h, sizeof(h), cudaMemcpyHostToDevice));
    const int grid = sms * 8;
    k_rcp<<<grid, kThreads>>>(d);
    k_bnd<<<grid, kThreads>>>(d);
    k_rnd<<<grid, kThreads>>>(d, n_rnd, 0x5eed0001ull);
    k_spc<<<1, 1>>>(d);
    k_e2e<<<grid, kThreads>>>(d, n_e2e, 0x5eed0002ull);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
    CK(cudaFree(d));
    printf("unary_obs");
    for (int k = 0; k < NCNT; k++) printf(" %s=%lld", kNames[k], (long long)h[k]);  // (first_bad_e2e: -1 = none)
    printf("\n");
    return 0;
}
