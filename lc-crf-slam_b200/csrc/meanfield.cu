// meanfield.cu -- the DenseCRF driver on the device.
// Replaces DenseCRF::startInference/stepInference (Thirdparty/DenseCRF/include/densecrf_base.h:78-91),
// DenseCRF3D<M>::expAndNormalize + fast_exp (densecrf3d.h:51-98), stepInit (:155-158),
// buildMap (:137-151) and setUnaryEnergyFromLabel (:108-130).
#include "engine.cuh"

namespace lccrf {

namespace {

// very_fast_exp / fast_exp, densecrf3d.h:51-67 -- operation for operation (a polynomial on a
// range-reduced argument followed by repeated squaring), NOT __expf: MAP near-ties follow the
// reference only if every rounding does.  The range-reduction thresholds are double constants.
__device__ __forceinline__ float very_fast_exp(float x) {
    float p = 0.0001413161f;
    p = __fsub_rn(0.0013298820f, __fmul_rn(x, p));
    p = __fsub_rn(0.0083013598f, __fmul_rn(x, p));
    p = __fsub_rn(0.0416573475f, __fmul_rn(x, p));
    p = __fsub_rn(0.1666653019f, __fmul_rn(x, p));
    p = __fsub_rn(0.4999999206f, __fmul_rn(x, p));
    p = __fsub_rn(0.9999999995f, __fmul_rn(x, p));
    return __fsub_rn(1.0f, __fmul_rn(x, p));
}

// The reference compares the float argument with DOUBLE thresholds (0.69*2*2*2 etc., densecrf3d.h:60-62).  For a
// float x and a double c:  (double)x > c  <=>  x > fl(c), fl(c) = the largest float <= c (no float lies strictly
// between fl(c) and c), so the comparisons run in fp32 with constants the compiler folds.  Dividing by 8, 4, 2 is
// a multiplication by 0.125, 0.25, 0.5: scaling by a power of two rounds identically either way.
__device__ __forceinline__ float float_at_or_below(double c) {
    float t = (float)c;
    if ((double)t > c) t = __int_as_float(__float_as_int(t) - 1);  // c > 0 here
    return t;
}

__device__ __forceinline__ float fast_exp(float x) {
    bool lessZero = true;
    if (x < 0) {
        lessZero = false;
        x = -x;
    }
    if (x > 20) return 0;
    const float t3 = float_at_or_below(0.69 * 2 * 2 * 2), t2 = float_at_or_below(0.69 * 2 * 2), t1 = float_at_or_below(0.69);
    int mult = 0;
    while (x > t3) {
        mult += 3;
        x = __fmul_rn(x, 0.125f);
    }
    while (x > t2) {
        mult += 2;
        x = __fmul_rn(x, 0.25f);
    }
    while (x > t1) {
        mult++;
        x = __fmul_rn(x, 0.5f);
    }
    x = very_fast_exp(x);
    while (mult) {
        mult--;
        x = __fmul_rn(x, x);
    }
    return lessZero ? __fdiv_rn(1.0f, x) : x;
}

// expAndNormalize, densecrf3d.h:71-98; one thread per point.  fast_exp is recomputed instead of
// buffered for run-time L (it is deterministic), kept in registers for L == 2.
template <int LT>
__global__ void __launch_bounds__(kThreads)
k_exp_normalize(float *__restrict__ out, const float *__restrict__ in, int NT, int L_rt, float scale, float relax) {
    const int L = LT > 0 ? LT : L_rt;
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= NT) return;
    const float *b = in + (size_t)i * L;
    float *a = out + (size_t)i * L;
    float mx = __fmul_rn(scale, b[0]);
    for (int j = 1; j < L; j++) {
        float s = __fmul_rn(scale, b[j]);
        if (mx < s) mx = s;
    }
    float tt = 0.f;
    if (LT == 2) {
        float v0 = fast_exp(__fsub_rn(__fmul_rn(scale, b[0]), mx));
        float v1 = fast_exp(__fsub_rn(__fmul_rn(scale, b[1]), mx));
        tt = __fadd_rn(__fadd_rn(tt, v0), v1);
        v0 = __fdiv_rn(v0, tt);
        v1 = __fdiv_rn(v1, tt);
        if (relax == 1.0f) {
            a[0] = v0;
            a[1] = v1;
        } else {
            const float om = __fsub_rn(1.0f, relax);
            a[0] = __fadd_rn(__fmul_rn(om, a[0]), __fmul_rn(relax, v0));
            a[1] = __fadd_rn(__fmul_rn(om, a[1]), __fmul_rn(relax, v1));
        }
        return;
    }
    for (int j = 0; j < L; j++) tt = __fadd_rn(tt, fast_exp(__fsub_rn(__fmul_rn(scale, b[j]), mx)));
    const float om = __fsub_rn(1.0f, relax);
    for (int j = 0; j < L; j++) {
        float v = __fdiv_rn(fast_exp(__fsub_rn(__fmul_rn(scale, b[j]), mx)), tt);
        a[j] = relax == 1.0f ? v : __fadd_rn(__fmul_rn(om, a[j]), __fmul_rn(relax, v));
    }
}

__global__ void __launch_bounds__(kThreads)
k_unary_from_label(float *__restrict__ unary, const short *__restrict__ label, int NT, int L, float u_energy,
                   const float *__restrict__ n_en, const float *__restrict__ p_en, int *__restrict__ status) {
    const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (t >= (long long)NT * L) return;
    const int i = (int)(t / L), m = (int)(t - (long long)i * L);
    int lab = label[i];
    if (status && (lab < -1 || lab >= L)) {  // the tables have L entries: report, and read the label as unknown
        if (m == 0) atomicOr(status, 32);
        lab = -1;
    }
    float v;
    if (lab == -1) v = u_energy;                       // densecrf3d.h:118-121
    else v = (m == lab) ? p_en[lab] : n_en[lab];      // :123-126
    unary[t] = v;
}

__global__ void __launch_bounds__(kThreads) k_negate(float *__restrict__ out, const float *__restrict__ in, long long n) {
    const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (t < n) out[t] = -in[t];  // stepInit, densecrf3d.h:155-158
}

__global__ void __launch_bounds__(kThreads)
k_build_map(short *__restrict__ map, const float *__restrict__ Q, int NT, int L) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= NT) return;
    const float *p = Q + (size_t)i * L;
    float mx = p[0];
    short imx = 0;
    for (int m = 1; m < L; m++)
        if (mx < p[m]) {  // strict: first maximum wins, densecrf3d.h:144-147
            mx = p[m];
            imx = (short)m;
        }
    map[i] = imx;
}

__global__ void __launch_bounds__(kThreads)
k_axpy_norm(float *__restrict__ out, const float *__restrict__ tmp, const float *__restrict__ norm, float w, int NT, int L) {
    const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (t >= (long long)NT * L) return;
    const int i = (int)(t / L);
    out[t] = __fadd_rn(out[t], __fmul_rn(__fmul_rn(w, norm[i]), tmp[t]));  // pairwise3d.h:75-77
}

// ---- fused point pass, L == 2: for every point, slice all K lattices (permutohedral_cpu.h:684-694), apply the
// Potts weights (pairwise3d.h:73-78) onto -unary (densecrf3d.h:155-158) and normalise (densecrf3d.h:71-98); same
// operation order as the unfused kernels, so the result is bit-identical
struct MfLat {
    const int *offset;
    const float *bary;
    const float2 *val;
    const float *norm;
    float w, alpha;
    int D;
};
struct MfArgs {
    int K;
    MfLat lat[LCCRF_MAX_K];
};

// expAndNormalize for two labels (densecrf3d.h:71-98) + optional buildMap (:137-151).  The label holding the maximum
// has the argument n - mx = +-0 (finite inputs) and fast_exp(+-0) is exactly 1.0f (very_fast_exp(0) = 1, 1/1 = 1), so the
// range-reduction loops of fast_exp run once per point, for the other label only; a non-zero argument of the maximum
// (inf - inf = NaN) still takes the full path, so the result is the reference's in every case.
__device__ __forceinline__ void softmax2_store(float n0, float n1, float2 *__restrict__ cur, short *__restrict__ map,
                                               int i, float relax) {
    const bool m0 = !(n0 < n1);  // mx = n0; if (mx < n1) mx = n1
    const float mx = m0 ? n0 : n1;
    const float a0 = __fsub_rn(n0, mx), a1 = __fsub_rn(n1, mx);
    const float am = m0 ? a0 : a1, ao = m0 ? a1 : a0;
    const float eo = fast_exp(ao);
    float em = 1.0f;
    if (!(am == 0.0f)) em = fast_exp(am);
    float v0 = m0 ? em : eo, v1 = m0 ? eo : em;
    const float tt = __fadd_rn(__fadd_rn(0.0f, v0), v1);
    v0 = __fdiv_rn(v0, tt);
    v1 = __fdiv_rn(v1, tt);
    if (relax != 1.0f) {
        const float2 old = cur[i];
        const float om = __fsub_rn(1.0f, relax);
        v0 = __fadd_rn(__fmul_rn(om, old.x), __fmul_rn(relax, v0));
        v1 = __fadd_rn(__fmul_rn(om, old.y), __fmul_rn(relax, v1));
    }
    cur[i] = make_float2(v0, v1);
    if (map) map[i] = (v0 < v1) ? 1 : 0;  // buildMap: strict <, first maximum wins
}

__global__ void __launch_bounds__(kThreads)
k_mf_point_l2(MfArgs a, const float2 *__restrict__ unary, float2 *__restrict__ cur, short *__restrict__ map, int NT,
              float relax) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= NT) return;
    const float2 u = __ldg(unary + i);
    float n0 = -u.x, n1 = -u.y;
    for (int k = 0; k < a.K; k++) {
        const MfLat &lt = a.lat[k];
        float s0 = 0.0f, s1 = 0.0f;
        for (int r = 0; r < lt.D; r++) {
            const int id = __ldg(lt.offset + (size_t)i * lt.D + r);
            const float wa = __fmul_rn(__ldg(lt.bary + (size_t)i * lt.D + r), lt.alpha);
            const float2 v = __ldg(lt.val + id);
            s0 = __fadd_rn(s0, __fmul_rn(wa, v.x));
            s1 = __fadd_rn(s1, __fmul_rn(wa, v.y));
        }
        const float wn = __fmul_rn(lt.w, __ldg(lt.norm + i));
        n0 = __fadd_rn(n0, __fmul_rn(wn, s0));
        n1 = __fadd_rn(n1, __fmul_rn(wn, s1));
    }
    softmax2_store(n0, n1, cur, map, i, relax);
}

// the SLAM / image shapes: two lattices with compile-time vertex counts per point.  Same operations in the same
// order as the generic kernel, but every index, weight and vertex value is requested before the first use
// (6 + 6 + 6 independent loads per point instead of a dependent load per loop trip) and nothing loops at run time.
template <int D0, int D1>
__global__ void __launch_bounds__(kThreads)
k_mf_point_l2_k2(MfArgs a, const float2 *__restrict__ unary, float2 *__restrict__ cur, short *__restrict__ map, int NT,
                 float relax) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= NT) return;
    int id0[D0], id1[D1];
    float w0[D0], w1[D1];
#pragma unroll
    for (int r = 0; r < D0; r++) id0[r] = __ldg(a.lat[0].offset + (size_t)i * D0 + r);
#pragma unroll
    for (int r = 0; r < D1; r++) id1[r] = __ldg(a.lat[1].offset + (size_t)i * D1 + r);
#pragma unroll
    for (int r = 0; r < D0; r++) w0[r] = __ldg(a.lat[0].bary + (size_t)i * D0 + r);
#pragma unroll
    for (int r = 0; r < D1; r++) w1[r] = __ldg(a.lat[1].bary + (size_t)i * D1 + r);
    const float2 u = __ldg(unary + i);
    const float nm0 = __ldg(a.lat[0].norm + i), nm1 = __ldg(a.lat[1].norm + i);
    float2 v0[D0], v1[D1];
#pragma unroll
    for (int r = 0; r < D0; r++) v0[r] = __ldg(a.lat[0].val + id0[r]);
#pragma unroll
    for (int r = 0; r < D1; r++) v1[r] = __ldg(a.lat[1].val + id1[r]);
    float n0 = -u.x, n1 = -u.y;
    {
        float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
        for (int r = 0; r < D0; r++) {
            const float wa = __fmul_rn(w0[r], a.lat[0].alpha);
            s0 = __fadd_rn(s0, __fmul_rn(wa, v0[r].x));
            s1 = __fadd_rn(s1, __fmul_rn(wa, v0[r].y));
        }
        const float wn = __fmul_rn(a.lat[0].w, nm0);
        n0 = __fadd_rn(n0, __fmul_rn(wn, s0));
        n1 = __fadd_rn(n1, __fmul_rn(wn, s1));
    }
    {
        float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
        for (int r = 0; r < D1; r++) {
            const float wa = __fmul_rn(w1[r], a.lat[1].alpha);
            s0 = __fadd_rn(s0, __fmul_rn(wa, v1[r].x));
            s1 = __fadd_rn(s1, __fmul_rn(wa, v1[r].y));
        }
        const float wn = __fmul_rn(a.lat[1].w, nm1);
        n0 = __fadd_rn(n0, __fmul_rn(wn, s0));
        n1 = __fadd_rn(n1, __fmul_rn(wn, s1));
    }
    softmax2_store(n0, n1, cur, map, i, relax);
}

}  // namespace

int mf_point_pass_l2(Ctx *ctx, Batch &b, const float *const *values, float relax, bool with_map) {
    if (b.NT == 0) return LCCRF_OK;
    MfArgs a;
    a.K = (int)b.lat.size();
    for (int k = 0; k < a.K; k++) {
        const LatticeSet *ls = b.lat[k];
        a.lat[k].offset = ls->offset;
        a.lat[k].bary = ls->bary;
        a.lat[k].val = (const float2 *)values[k];
        a.lat[k].norm = ls->norm;
        a.lat[k].w = ls->w;
        a.lat[k].alpha = ls->alpha;
        a.lat[k].D = ls->D;
    }
    LCCRF_KERNEL(ctx, "k_mf_point_l2");
    const int grid = cdiv(b.NT, kThreads);
    short *mp = with_map ? b.map : nullptr;
    if (a.K == 2 && a.lat[0].D == 3 && a.lat[1].D == 3)        // SLAM: appearance + smoothness, both 2-D features
        k_mf_point_l2_k2<3, 3><<<grid, kThreads, 0, ctx->stream>>>(a, (const float2 *)b.unary, (float2 *)b.cur, mp, b.NT, relax);
    else if (a.K == 2 && a.lat[0].D == 3 && a.lat[1].D == 6)   // image: Gaussian (x, y) + bilateral (x, y, r, g, b)
        k_mf_point_l2_k2<3, 6><<<grid, kThreads, 0, ctx->stream>>>(a, (const float2 *)b.unary, (float2 *)b.cur, mp, b.NT, relax);
    else
        k_mf_point_l2<<<grid, kThreads, 0, ctx->stream>>>(a, (const float2 *)b.unary, (float2 *)b.cur, mp, b.NT, relax);
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int launch_axpy_norm(Ctx *ctx, float *out, const float *tmp, const float *norm, float w, int NT, int L) {
    if (NT == 0) return LCCRF_OK;
    { LCCRF_KERNEL(ctx, "k_axpy_norm"); k_axpy_norm<<<cdiv((long long)NT * L, kThreads), kThreads, 0, ctx->stream>>>(out, tmp, norm, w, NT, L); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int mf_unary_from_label(Ctx *ctx, float *unary, const short *label_dev, int NT, int L, float u_energy,
                        const float *n_en_dev, const float *p_en_dev, int *status) {
    if (NT == 0) return LCCRF_OK;
    { LCCRF_KERNEL(ctx, "k_unary_from_label"); k_unary_from_label<<<cdiv((long long)NT * L, kThreads), kThreads, 0, ctx->stream>>>(unary, label_dev, NT, L, u_energy,
                                                                                       n_en_dev, p_en_dev, status); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int mf_exp_and_normalize(Ctx *ctx, float *out, const float *in, int NT, int L, float scale, float relax) {
    if (NT == 0) return LCCRF_OK;
    const int grid = cdiv(NT, kThreads);
    if (L == 2) { LCCRF_KERNEL(ctx, "k_exp_normalize"); k_exp_normalize<2><<<grid, kThreads, 0, ctx->stream>>>(out, in, NT, L, scale, relax); }
    else { LCCRF_KERNEL(ctx, "k_exp_normalize"); k_exp_normalize<0><<<grid, kThreads, 0, ctx->stream>>>(out, in, NT, L, scale, relax); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int mf_negate(Ctx *ctx, float *out, const float *in, long long n) {
    if (n == 0) return LCCRF_OK;
    { LCCRF_KERNEL(ctx, "k_negate"); k_negate<<<cdiv(n, kThreads), kThreads, 0, ctx->stream>>>(out, in, n); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

// startInference: Q = softmax(-U)   densecrf_base.h:78-80
int mf_start(Ctx *ctx, Batch &b) { return mf_exp_and_normalize(ctx, b.cur, b.unary, b.NT, b.L, -1.0f, 1.0f); }

// stepInference   densecrf_base.h:82-91
int mf_step(Ctx *ctx, Batch &b, float relax) {
    if (b.NT == 0) return LCCRF_OK;
    if (b.L == 2 && !b.lat.empty() && ctx->opt_fused) {
        // splat + blur of every lattice from the same Q, then ONE point pass
        // (odd lattices on the aux branch: the filters of different lattices are independent)
        const float *vals[LCCRF_MAX_K];
        const bool par = b.lat.size() > 1;
        if (par) LCCRF_TRY(ctx_fork(ctx));
        for (size_t k = 0; k < b.lat.size(); k++) {
            AuxScope aux(ctx, par && (k & 1));
            LCCRF_TRY(filter_splat_blur(ctx, b, b.lat[k], b.cur, 2, &vals[k]));
        }
        if (par) LCCRF_TRY(ctx_join(ctx));
        return mf_point_pass_l2(ctx, b, vals, relax, false);
    }
    if (b.lat.empty()) LCCRF_TRY(mf_negate(ctx, b.next, b.unary, (long long)b.NT * b.L));
    for (size_t k = 0; k < b.lat.size(); k++) LCCRF_TRY(mf_apply_fused(ctx, b, b.lat[k], b.cur, b.next, b.unary, k == 0));
    return mf_exp_and_normalize(ctx, b.cur, b.next, b.NT, b.L, 1.0f, relax);
}

int mf_build_map(Ctx *ctx, Batch &b) {
    if (b.NT == 0) return LCCRF_OK;
    { LCCRF_KERNEL(ctx, "k_build_map"); k_build_map<<<cdiv(b.NT, kThreads), kThreads, 0, ctx->stream>>>(b.map, b.cur, b.NT, b.L); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

}  // namespace lccrf
