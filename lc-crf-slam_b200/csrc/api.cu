// api.cu -- the extern "C" boundary (include/lccrf.h) and the host-side engine objects.
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "engine.cuh"

namespace lccrf {

static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

// ------------------------------------------------------------------ memory
int dev_alloc(Ctx *ctx, void **p, size_t bytes, bool zero) {
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMallocAsync(p, bytes, ctx->stream);
    if (e != cudaSuccess) return fail(LCCRF_ERR_CUDA, std::string("cudaMallocAsync: ") + cudaGetErrorString(e));
    if (zero) {
        e = cudaMemsetAsync(*p, 0, bytes, ctx->stream);
        if (e != cudaSuccess) return fail(LCCRF_ERR_CUDA, std::string("cudaMemsetAsync: ") + cudaGetErrorString(e));
    }
    return LCCRF_OK;
}

void dev_free(Ctx *ctx, void *p) {
    if (p) cudaFreeAsync(p, ctx->stream);
}

int ctx_scratch(Ctx *ctx, Ctx::Scratch &s, size_t bytes, bool pinned) {
    if (bytes <= s.bytes && s.p) return LCCRF_OK;
    size_t want = bytes + bytes / 4 + 256;
    ctx->scratch_gen++;
    // growth is rare (first use of a shape) and may happen on either branch: order it against both streams
    if (s.p) {
        cudaStreamSynchronize(ctx->stream);
        if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
    }
    if (pinned) {
        if (s.p) cudaFreeHost(s.p);
        s.p = nullptr;
        s.bytes = 0;
        LCCRF_CUDA(cudaHostAlloc(&s.p, want, cudaHostAllocDefault));
    } else {
        if (s.p) cudaFree(s.p);
        s.p = nullptr;
        s.bytes = 0;
        LCCRF_CUDA(cudaMalloc(&s.p, want));
    }
    s.bytes = want;
    return LCCRF_OK;
}

bool ctx_concurrent(const Ctx *ctx) { return ctx->opt_concurrent && !ctx->opt_profile && ctx->aux_stream; }

int ctx_fork(Ctx *ctx) {
    if (!ctx_concurrent(ctx)) return LCCRF_OK;
    LCCRF_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    LCCRF_CUDA(cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_fork, 0));
    return LCCRF_OK;
}

int ctx_join(Ctx *ctx) {
    if (!ctx_concurrent(ctx)) return LCCRF_OK;
    LCCRF_CUDA(cudaEventRecord(ctx->ev_join, ctx->aux_stream));
    LCCRF_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    return LCCRF_OK;
}

bool uniform_camera(const float *kf_intr, const float *kf_bounds, int nKF, float *cam8) {
    if (nKF <= 0 || !kf_intr || !kf_bounds) return false;
    for (int k = 1; k < nKF; k++)
        if (memcmp(kf_intr + 4 * (size_t)k, kf_intr, 16) != 0 || memcmp(kf_bounds + 4 * (size_t)k, kf_bounds, 16) != 0)
            return false;
    memcpy(cam8, kf_intr, 16);
    memcpy(cam8 + 4, kf_bounds, 16);
    return true;
}

static void scratch_release(Ctx *ctx, Ctx::Scratch &s, bool pinned) {
    (void)ctx;
    if (!s.p) return;
    if (pinned) cudaFreeHost(s.p);
    else cudaFree(s.p);
    s.p = nullptr;
    s.bytes = 0;
}

// device status word -> error code (bits: 1 lattice key range, 2 index out of range, 4 visible point without
// observations, 8 a point twice in one delta list, 16 observation pool exhausted, 32 label outside [-1, L))
int decode_status(int st) {
    if (st & 1) return fail(LCCRF_ERR_RANGE, "lattice key outside the reference's short range (permutohedral_cpu.h:373)");
    if (st & 2) return fail(LCCRF_ERR_ARG, "an observation, keyframe, feature or point index is outside its table");
    if (st & 4) return fail(LCCRF_ERR_ARG, "a visible map point has no observations (Tracking.cc:1858 drops such points before the CRF)");
    if (st & 8) return fail(LCCRF_ERR_ARG, "a point appears twice in one list of a map delta (split it over several deltas)");
    if (st & 16) return fail(LCCRF_ERR_STATE, "observation pool exhausted: call lccrf_map_reserve_observations and repeat the step");
    if (st & 32) return fail(LCCRF_ERR_ARG, "a label is outside [-1, L)");
    return LCCRF_OK;
}

int check_status(Ctx *ctx) {  // synchronises
    LCCRF_CUDA(cudaMemcpyAsync(ctx->h_status, ctx->d_status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    if (*ctx->h_status) {
        cudaMemsetAsync(ctx->d_status, 0, sizeof(int), ctx->stream);
        return decode_status(*ctx->h_status);
    }
    return LCCRF_OK;
}

int batch_init(Ctx *ctx, Batch &b, int B, const int *prob_ptr, int L, bool with_state) {
    b.ctx = ctx;
    b.B = B;
    b.L = L;
    b.h_prob_ptr.assign(prob_ptr, prob_ptr + B + 1);
    if (b.h_prob_ptr[0] != 0) return fail(LCCRF_ERR_ARG, "prob_ptr[0] must be 0");
    b.maxN = 0;
    for (int i = 0; i < B; i++) {
        int n = b.h_prob_ptr[i + 1] - b.h_prob_ptr[i];
        if (n < 0) return fail(LCCRF_ERR_ARG, "prob_ptr must be non-decreasing");
        if (n > b.maxN) b.maxN = n;
    }
    if (b.maxN > (1 << 22)) return fail(LCCRF_ERR_ARG, "more than 2^22 points in one problem (fixed-point splat range)");
    b.NT = b.h_prob_ptr[B];
    b.fused_blur = B >= 2 || b.maxN <= kFusedBlurMaxN;
    LCCRF_TRY(dev_alloc(ctx, (void **)&b.prob_ptr, (size_t)(B + 1) * sizeof(int)));
    LCCRF_CUDA(cudaMemcpyAsync(b.prob_ptr, b.h_prob_ptr.data(), (size_t)(B + 1) * sizeof(int), cudaMemcpyHostToDevice,
                               ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    if (with_state) {
        const size_t n = (size_t)(b.NT > 0 ? b.NT : 1) * L * sizeof(float);
        LCCRF_TRY(dev_alloc(ctx, (void **)&b.unary, n));
        LCCRF_TRY(dev_alloc(ctx, (void **)&b.cur, n));
        LCCRF_TRY(dev_alloc(ctx, (void **)&b.next, n));
        LCCRF_TRY(dev_alloc(ctx, (void **)&b.tmp, n));
        LCCRF_TRY(dev_alloc(ctx, (void **)&b.map, (size_t)(b.NT > 0 ? b.NT : 1) * sizeof(short)));
    }
    return LCCRF_OK;
}

void batch_release(Ctx *ctx, Batch &b) {
    for (auto *ls : b.lat) lattice_set_destroy(ctx, ls);
    b.lat.clear();
    dev_free(ctx, b.prob_ptr);
    dev_free(ctx, b.unary);
    dev_free(ctx, b.cur);
    dev_free(ctx, b.next);
    dev_free(ctx, b.tmp);
    dev_free(ctx, b.map);
    b.prob_ptr = nullptr;
    b.unary = b.cur = b.next = b.tmp = nullptr;
    b.map = nullptr;
}

void graph_drop(GraphReplay &g) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    g.exec = nullptr;
    g.same_shape_runs = 0;
}

bool graph_will_capture(const Ctx *ctx, const GraphReplay &g) {
    return ctx->opt_graphs && !ctx->opt_profile && !g.exec && g.same_shape_runs > 0;
}

int graph_run(Ctx *ctx, GraphReplay &g, const std::function<int()> &enqueue) {
    if (!ctx->opt_graphs || ctx->opt_profile) return enqueue();
    if (g.exec && g.gen != ctx->scratch_gen) graph_drop(g);  // a scratch buffer moved since capture
    if (!g.exec && g.same_shape_runs == 0) {
        // A new shape: plain launches, no synchronisation.  A graph is only worth capturing for a shape that repeats,
        // so the capture waits for the second run of the same shape.
        g.same_shape_runs = 1;
        return enqueue();
    }
    if (!g.exec) {
        // make sure every scratch buffer has its final size before capture (no allocation inside the graph)
        const uint64_t l0 = ctx->launches;
        LCCRF_TRY(enqueue());
        LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
        const uint64_t per_run = ctx->launches - l0;
        cudaGraph_t cg = nullptr;
        LCCRF_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue();
        cudaError_t e = cudaStreamEndCapture(ctx->stream, &cg);
        ctx->launches -= per_run;  // the capture pass launched nothing
        if (rc != LCCRF_OK) {
            if (cg) cudaGraphDestroy(cg);
            return rc;
        }
        if (e != cudaSuccess) return fail(LCCRF_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(e));
        e = cudaGraphInstantiate(&g.exec, cg, 0);
        cudaGraphDestroy(cg);
        if (e != cudaSuccess) return fail(LCCRF_ERR_CUDA, std::string("graph instantiate: ") + cudaGetErrorString(e));
        g.launches = per_run;
        g.gen = ctx->scratch_gen;
        return LCCRF_OK;  // the warm-up pass above already produced this call's results
    }
    LCCRF_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
    ctx->launches += g.launches;
    return LCCRF_OK;
}

}  // namespace lccrf

using namespace lccrf;

// ------------------------------------------------------------------ opaque handle types (lccrf_ctx: engine.cuh)
struct lccrf_lattice {
    Ctx *ctx = nullptr;
    Batch b;
    LatticeSet *ls = nullptr;
    int V = 0;
    float *io = nullptr;  // device in/out buffer for filter calls
    size_t io_bytes = 0;
};

struct lccrf_crf {
    Ctx *ctx = nullptr;
    Batch b;
    bool started = false;
    float *h_prob = nullptr;  // pinned
    short *h_map = nullptr;   // pinned
    bool prob_fresh = false, map_fresh = false, map_built = false;
    float *d_energies = nullptr;  // n_en[L], p_en[L]
};

extern "C" {

const char *lccrf_version(void) { return "lccrf-b200 0.1 (sm_100a)"; }
const char *lccrf_last_error(void) { return g_err.c_str(); }

int lccrf_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int lccrf_ctx_create(int device, lccrf_ctx **out) {
    if (!out) return fail(LCCRF_ERR_ARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(LCCRF_ERR_CUDA, std::string("no CUDA device available (there is no CPU fallback): ") +
                                        (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device < 0 || device >= n) return fail(LCCRF_ERR_ARG, "device index out of range");
    LCCRF_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    LCCRF_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(LCCRF_ERR_CUDA, std::string("liblccrf is built for sm_100a only; device is ") + prop.name);
    auto *h = new lccrf_ctx();
    h->c.device = device;
    cudaError_t es = cudaStreamCreateWithFlags(&h->c.stream, cudaStreamNonBlocking);
    if (es != cudaSuccess) {
        delete h;
        return fail(LCCRF_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(es));
    }
    h->c.own_stream = true;
    if (cudaStreamCreateWithFlags(&h->c.aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->c.ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->c.ev_join, cudaEventDisableTiming) != cudaSuccess) {
        delete h;
        return fail(LCCRF_ERR_CUDA, "aux stream / event creation failed");
    }
    for (int i = 0; i < 2; i++)
        if (cudaStreamCreateWithFlags(&h->c.sub_stream[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&h->c.ev_sub_fork[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&h->c.ev_sub_join[i], cudaEventDisableTiming) != cudaSuccess) {
            delete h;
            return fail(LCCRF_ERR_CUDA, "sub stream / event creation failed");
        }
    // keep freed blocks cached in the stream-ordered pool: per-frame CRF objects allocate and free constantly
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    if (cudaMalloc((void **)&h->c.d_status, sizeof(int)) != cudaSuccess ||
        cudaMemset(h->c.d_status, 0, sizeof(int)) != cudaSuccess ||
        cudaHostAlloc((void **)&h->c.h_status, sizeof(int), cudaHostAllocDefault) != cudaSuccess) {
        delete h;
        return fail(LCCRF_ERR_CUDA, "status word allocation failed");
    }
    *out = h;
    return LCCRF_OK;
}

void lccrf_ctx_destroy(lccrf_ctx *h) {
    if (!h) return;
    Ctx *c = &h->c;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->aux_stream) cudaStreamSynchronize(c->aux_stream);
    for (auto &bs : c->bs) {
        for (auto &s : bs.hash_keys) scratch_release(c, s, false);
        scratch_release(c, bs.hash_first, false);
        scratch_release(c, bs.hash_id, false);
        scratch_release(c, bs.ent_slot, false);
        scratch_release(c, bs.ids_status, false);
    }
    scratch_release(c, c->misc, false);
    scratch_release(c, c->feat, false);
    scratch_release(c, c->dev_io, false);
    scratch_release(c, c->pinned_in, true);
    scratch_release(c, c->pinned_out, true);
    cudaStreamSynchronize(c->stream);
    cudaFree(c->d_status);
    cudaFreeHost(c->h_status);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    for (int i = 0; i < 2; i++) {
        if (c->sub_stream[i]) cudaStreamDestroy(c->sub_stream[i]);
        if (c->ev_sub_fork[i]) cudaEventDestroy(c->ev_sub_fork[i]);
        if (c->ev_sub_join[i]) cudaEventDestroy(c->ev_sub_join[i]);
    }
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete h;
}

int lccrf_ctx_set_stream(lccrf_ctx *h, void *cuda_stream) {
    if (!h) return fail(LCCRF_ERR_ARG, "ctx is NULL");
    Ctx *c = &h->c;
    LCCRF_CUDA(cudaSetDevice(c->device));
    LCCRF_CUDA(cudaStreamSynchronize(c->stream));
    if (c->own_stream) cudaStreamDestroy(c->stream);
    if (cuda_stream) {
        c->stream = (cudaStream_t)cuda_stream;
        c->own_stream = false;
    } else {
        LCCRF_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    return LCCRF_OK;
}

int lccrf_ctx_sync(lccrf_ctx *h) {
    if (!h) return fail(LCCRF_ERR_ARG, "ctx is NULL");
    LCCRF_CUDA(cudaStreamSynchronize(h->c.stream));
    return LCCRF_OK;
}

uint64_t lccrf_ctx_kernel_launches(const lccrf_ctx *h) { return h ? h->c.launches : 0; }

int lccrf_ctx_build_scratch_in_use(lccrf_ctx *h, long long *slots) {
    if (!h || !slots) return fail(LCCRF_ERR_ARG, "NULL argument");
    return build_scratch_in_use(&h->c, slots);
}

int lccrf_ctx_set_option(lccrf_ctx *h, const char *name, int value) {
    if (!h || !name) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx &c = h->c;
    // switches that select the launch sequence (kernel set, branch structure): captured graphs hold the other sequence,
    // so a change makes every one of them stale
    const struct {
        const char *name;
        int *opt;
    } sequence[] = {{"fused", &c.opt_fused}, {"ordered_splat", &c.opt_ordered_splat}, {"bulk_blur", &c.opt_bulk_blur},
                    {"concurrent", &c.opt_concurrent}, {"split_splat", &c.opt_split_splat}};
    for (const auto &s : sequence)
        if (!strcmp(name, s.name)) {
            if (*s.opt != (value ? 1 : 0)) c.scratch_gen++;
            *s.opt = value ? 1 : 0;
            return LCCRF_OK;
        }
    if (!strcmp(name, "graphs")) c.opt_graphs = value;
    else if (!strcmp(name, "profile")) c.opt_profile = value;
    else if (!strcmp(name, "map_slack")) c.opt_map_slack = value < 0 ? 0 : value;
    else if (!strcmp(name, "trace")) c.opt_trace = value;
    else return fail(LCCRF_ERR_ARG, std::string("unknown option ") + name);
    return LCCRF_OK;
}

int lccrf_ctx_profile_report(lccrf_ctx *h, char *buf, int cap) {
    if (!h || !buf || cap < 1) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *c = &h->c;
    LCCRF_CUDA(cudaSetDevice(c->device));
    LCCRF_CUDA(cudaStreamSynchronize(c->stream));
    std::vector<std::string> names;
    std::vector<double> ms;
    std::vector<long long> cnt;
    for (auto &r : c->prof) {
        float t = 0.f;
        cudaEventElapsedTime(&t, r.a, r.b);
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
        size_t k = 0;
        for (; k < names.size(); k++)
            if (names[k] == r.name) break;
        if (k == names.size()) {
            names.push_back(r.name);
            ms.push_back(0);
            cnt.push_back(0);
        }
        ms[k] += t;
        cnt[k]++;
    }
    c->prof.clear();
    std::string out;
    char line[256];
    for (size_t k = 0; k < names.size(); k++) {
        snprintf(line, sizeof(line), "%s %lld %.6f\n", names[k].c_str(), cnt[k], ms[k]);
        out += line;
    }
    strncpy(buf, out.c_str(), (size_t)cap - 1);
    buf[cap - 1] = 0;
    return (int)names.size();
}

// ------------------------------------------------------------------ lattice
int lccrf_lattice_create(lccrf_ctx *h, const float *features, int d, int N, lccrf_lattice **out) {
    if (!h || !out || (N > 0 && !features)) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (N < 0) return fail(LCCRF_ERR_ARG, "N < 0");
    *out = nullptr;
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    auto *lat = new lccrf_lattice();
    lat->ctx = ctx;
    int pp[2] = {0, N};
    int rc = batch_init(ctx, lat->b, 1, pp, 1, false);
    if (rc == LCCRF_OK) rc = lattice_set_create(ctx, lat->b, d, 1.0f, 0, &lat->ls);
    if (rc == LCCRF_OK) rc = ctx_scratch(ctx, ctx->feat, (size_t)(N > 0 ? N : 1) * d * sizeof(float));
    if (rc == LCCRF_OK && N > 0) {
        cudaError_t e = cudaMemcpyAsync(ctx->feat.p, features, (size_t)N * d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
    }
    if (rc == LCCRF_OK) rc = lattice_set_build(ctx, lat->b, lat->ls, (const float *)ctx->feat.p);
    if (rc == LCCRF_OK) {
        cudaError_t e = cudaMemcpyAsync(ctx->h_status, lat->ls->vbase + 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
        else lat->V = *ctx->h_status;
    }
    if (rc == LCCRF_OK) rc = check_status(ctx);
    if (rc != LCCRF_OK) {
        lccrf_lattice_destroy(lat);
        return rc;
    }
    *out = lat;
    return LCCRF_OK;
}

void lccrf_lattice_destroy(lccrf_lattice *lat) {
    if (!lat) return;
    cudaSetDevice(lat->ctx->device);
    if (lat->ls) lattice_set_destroy(lat->ctx, lat->ls);
    lat->ls = nullptr;
    batch_release(lat->ctx, lat->b);
    dev_free(lat->ctx, lat->io);
    delete lat;
}

int lccrf_lattice_sizes(const lccrf_lattice *lat, int *N, int *d, int *V) {
    if (!lat) return fail(LCCRF_ERR_ARG, "lattice is NULL");
    if (N) *N = lat->b.NT;
    if (d) *d = lat->ls->d;
    if (V) *V = lat->V;
    return LCCRF_OK;
}

int lccrf_lattice_export(const lccrf_lattice *lat, int *offset, float *bary, int *nbr) {
    if (!lat) return fail(LCCRF_ERR_ARG, "lattice is NULL");
    Ctx *ctx = lat->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const LatticeSet *ls = lat->ls;
    const size_t nent = (size_t)lat->b.NT * ls->D;
    // B == 1: global ids == reference ids (vbase[0] == 0)
    if (offset && nent) LCCRF_CUDA(cudaMemcpyAsync(offset, ls->offset, nent * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (bary && nent) LCCRF_CUDA(cudaMemcpyAsync(bary, ls->bary, nent * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (nbr && lat->V > 0) {
        for (int j = 0; j < ls->D; j++)
            LCCRF_CUDA(cudaMemcpyAsync(nbr + 2 * (size_t)j * lat->V, ls->nbr + (size_t)j * ls->Vcap,
                                       (size_t)lat->V * sizeof(int2), cudaMemcpyDeviceToHost, ctx->stream));
    }
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

int lccrf_lattice_filter_window(lccrf_lattice *lat, float *out, const float *in, int L, int in_offset, int out_offset,
                                int in_size, int out_size) {
    if (!lat || !out || !in) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (L < 1 || L > LCCRF_MAX_L) return fail(LCCRF_ERR_ARG, "L out of range");
    const int N = lat->b.NT;
    if (in_size == -1) in_size = N - in_offset;      // permutohedral_cpu.h:636-637
    if (out_size == -1) out_size = N - out_offset;
    if (in_offset < 0 || out_offset < 0 || in_size < 0 || out_size < 0 || (long long)in_offset + in_size > N ||
        (long long)out_offset + out_size > N)
        return fail(LCCRF_ERR_ARG, "filter window outside [0, N)");
    Ctx *ctx = lat->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)N * L;
    if (n == 0 || out_size == 0) return LCCRF_OK;
    LCCRF_TRY(lattice_set_ensure_L(ctx, lat->ls, L));
    if (lat->io_bytes < 2 * n * sizeof(float)) {
        dev_free(ctx, lat->io);
        lat->io = nullptr;
        lat->io_bytes = 0;
        LCCRF_TRY(dev_alloc(ctx, (void **)&lat->io, 2 * n * sizeof(float)));
        lat->io_bytes = 2 * n * sizeof(float);
    }
    float *d_in = lat->io, *d_out = lat->io + n;
    // points outside the input window contribute products of +-0, which leave the (+0-started) vertex sums untouched
    if (in_size != N) LCCRF_CUDA(cudaMemsetAsync(d_in, 0, n * sizeof(float), ctx->stream));
    if (in_size > 0)
        LCCRF_CUDA(cudaMemcpyAsync(d_in + (size_t)in_offset * L, in, (size_t)in_size * L * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_TRY(filter_full(ctx, lat->b, lat->ls, d_out, d_in, L));
    LCCRF_CUDA(cudaMemcpyAsync(out, d_out + (size_t)out_offset * L, (size_t)out_size * L * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

int lccrf_lattice_filter(lccrf_lattice *lat, float *out, const float *in, int L) {
    return lccrf_lattice_filter_window(lat, out, in, L, 0, 0, -1, -1);
}

int lccrf_lattice_debug_counters(const lccrf_lattice *lat, int *out8) {
    if (!lat || !out8) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = lat->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    LCCRF_CUDA(cudaMemcpyAsync(out8, lat->ls->row_counts, 8 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

// ------------------------------------------------------------------ dense CRF
int lccrf_crf_create(lccrf_ctx *h, int N, int L, lccrf_crf **out) {
    if (!h || !out) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (N < 0 || L < 1 || L > LCCRF_MAX_L) return fail(LCCRF_ERR_ARG, "N or L out of range");
    *out = nullptr;
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    auto *crf = new lccrf_crf();
    crf->ctx = ctx;
    int pp[2] = {0, N};
    int rc = batch_init(ctx, crf->b, 1, pp, L, true);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&crf->d_energies, 2 * (size_t)L * sizeof(float));
    if (rc == LCCRF_OK) {
        const size_t n = (size_t)(N > 0 ? N : 1);
        if (cudaHostAlloc((void **)&crf->h_prob, n * L * sizeof(float), cudaHostAllocDefault) != cudaSuccess ||
            cudaHostAlloc((void **)&crf->h_map, n * sizeof(short), cudaHostAllocDefault) != cudaSuccess)
            rc = fail(LCCRF_ERR_CUDA, "pinned result buffers: cudaHostAlloc failed");
    }
    if (rc != LCCRF_OK) {
        lccrf_crf_destroy(crf);
        return rc;
    }
    *out = crf;
    return LCCRF_OK;
}

void lccrf_crf_destroy(lccrf_crf *crf) {
    if (!crf) return;
    cudaSetDevice(crf->ctx->device);
    cudaStreamSynchronize(crf->ctx->stream);
    batch_release(crf->ctx, crf->b);
    dev_free(crf->ctx, crf->d_energies);
    if (crf->h_prob) cudaFreeHost(crf->h_prob);
    if (crf->h_map) cudaFreeHost(crf->h_map);
    delete crf;
}

int lccrf_crf_set_unary(lccrf_crf *crf, const float *unary) {
    if (!crf || (!unary && crf->b.NT > 0)) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)crf->b.NT * crf->b.L;
    if (n) LCCRF_CUDA(cudaMemcpyAsync(crf->b.unary, unary, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));  // the caller may free `unary` right away (densecrf3d.h:42 copies)
    return LCCRF_OK;
}

int lccrf_crf_set_unary_from_label(lccrf_crf *crf, const short *label, float u_energy, const float *n_energies,
                                   const float *p_energies) {
    if (!crf || !n_energies || !p_energies || (!label && crf->b.NT > 0)) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const int NT = crf->b.NT, L = crf->b.L;
    for (int i = 0; i < NT; i++)
        if (label[i] < -1 || label[i] >= L) return fail(LCCRF_ERR_ARG, "label outside [-1, L)");
    LCCRF_CUDA(cudaMemcpyAsync(crf->d_energies, n_energies, (size_t)L * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaMemcpyAsync(crf->d_energies + L, p_energies, (size_t)L * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if (NT > 0) {
        LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, (size_t)NT * sizeof(short)));
        LCCRF_CUDA(cudaMemcpyAsync(ctx->dev_io.p, label, (size_t)NT * sizeof(short), cudaMemcpyHostToDevice, ctx->stream));
        LCCRF_TRY(mf_unary_from_label(ctx, crf->b.unary, (const short *)ctx->dev_io.p, NT, L, u_energy, crf->d_energies,
                                      crf->d_energies + L));
    }
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

int lccrf_crf_set_unary_entry(lccrf_crf *crf, int idx, int m, float value) {
    if (!crf) return fail(LCCRF_ERR_ARG, "crf is NULL");
    if (idx < 0 || idx >= crf->b.NT || m < 0 || m >= crf->b.L) return fail(LCCRF_ERR_ARG, "index out of range");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    LCCRF_CUDA(cudaMemcpyAsync(crf->b.unary + (size_t)idx * crf->b.L + m, &value, sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

static int crf_add_lattice(lccrf_crf *crf, int d, float w, const float *feat_dev) {
    Ctx *ctx = crf->ctx;
    if ((int)crf->b.lat.size() >= LCCRF_MAX_K) return fail(LCCRF_ERR_ARG, "too many pairwise potentials");
    LatticeSet *ls = nullptr;
    LCCRF_TRY(lattice_set_create(ctx, crf->b, d, w, crf->b.L, &ls));
    int rc = lattice_set_build(ctx, crf->b, ls, feat_dev);
    if (rc == LCCRF_OK) rc = potts_norm(ctx, crf->b, ls);
    if (rc == LCCRF_OK) rc = check_status(ctx);
    if (rc != LCCRF_OK) {
        lattice_set_destroy(ctx, ls);
        return rc;
    }
    crf->b.lat.push_back(ls);
    return LCCRF_OK;
}

int lccrf_crf_add_potts(lccrf_crf *crf, const float *features, int d, float w) {
    if (!crf || (!features && crf->b.NT > 0)) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (d < 1 || d > LCCRF_MAX_D) return fail(LCCRF_ERR_ARG, "feature dimension must be in [1, LCCRF_MAX_D]");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)crf->b.NT * d;
    LCCRF_TRY(ctx_scratch(ctx, ctx->feat, (n ? n : 1) * sizeof(float)));
    if (n) LCCRF_CUDA(cudaMemcpyAsync(ctx->feat.p, features, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    return crf_add_lattice(crf, d, w, (const float *)ctx->feat.p);
}

int lccrf_crf_add_potts_image(lccrf_crf *crf, int W, int H, float w, float posdev, const void *img, int img_is_u8,
                              int F, float featuredev) {
    if (!crf) return fail(LCCRF_ERR_ARG, "crf is NULL");
    if (W < 0 || H < 0 || (long long)W * H != crf->b.NT) return fail(LCCRF_ERR_ARG, "W*H must equal N");
    if (F < 2 || F > LCCRF_MAX_D) return fail(LCCRF_ERR_ARG, "F must be in [2, LCCRF_MAX_D]");
    if (F > 2 && !img && crf->b.NT > 0) return fail(LCCRF_ERR_ARG, "image features required when F > 2");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t npx = (size_t)crf->b.NT;
    LCCRF_TRY(ctx_scratch(ctx, ctx->feat, (npx ? npx : 1) * F * sizeof(float)));
    const void *img_dev = nullptr;
    if (F > 2 && npx) {
        const size_t ib = npx * (F - 2) * (img_is_u8 ? 1 : sizeof(float));
        LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, ib));
        LCCRF_CUDA(cudaMemcpyAsync(ctx->dev_io.p, img, ib, cudaMemcpyHostToDevice, ctx->stream));
        img_dev = ctx->dev_io.p;
    }
    LCCRF_TRY(feat_image(ctx, (float *)ctx->feat.p, W, H, F, posdev, img_dev, img_is_u8, featuredev));
    return crf_add_lattice(crf, F, w, (const float *)ctx->feat.p);
}

int lccrf_crf_start(lccrf_crf *crf) {
    if (!crf) return fail(LCCRF_ERR_ARG, "crf is NULL");
    LCCRF_CUDA(cudaSetDevice(crf->ctx->device));
    LCCRF_TRY(mf_start(crf->ctx, crf->b));
    crf->started = true;
    crf->prob_fresh = false;
    return LCCRF_OK;
}

int lccrf_crf_step(lccrf_crf *crf, float relax) {
    if (!crf) return fail(LCCRF_ERR_ARG, "crf is NULL");
    if (!crf->started) return fail(LCCRF_ERR_STATE, "stepInference before startInference");
    LCCRF_CUDA(cudaSetDevice(crf->ctx->device));
    LCCRF_TRY(mf_step(crf->ctx, crf->b, relax));
    crf->prob_fresh = false;
    return LCCRF_OK;
}

int lccrf_crf_build_map(lccrf_crf *crf) {
    if (!crf) return fail(LCCRF_ERR_ARG, "crf is NULL");
    LCCRF_CUDA(cudaSetDevice(crf->ctx->device));
    LCCRF_TRY(mf_build_map(crf->ctx, crf->b));
    crf->map_built = true;
    crf->map_fresh = false;
    return LCCRF_OK;
}

static int crf_fetch(lccrf_crf *crf) {
    Ctx *ctx = crf->ctx;
    const size_t n = (size_t)crf->b.NT;
    bool any = false;
    if (!crf->prob_fresh && n) {
        LCCRF_CUDA(cudaMemcpyAsync(crf->h_prob, crf->b.cur, n * crf->b.L * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        any = true;
    }
    if (crf->map_built && !crf->map_fresh && n) {
        LCCRF_CUDA(cudaMemcpyAsync(crf->h_map, crf->b.map, n * sizeof(short), cudaMemcpyDeviceToHost, ctx->stream));
        any = true;
    }
    if (any) LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    crf->prob_fresh = true;
    if (crf->map_built) crf->map_fresh = true;
    return LCCRF_OK;
}

int lccrf_crf_inference(lccrf_crf *crf, int n_iterations, int with_map, float relax) {
    if (!crf) return fail(LCCRF_ERR_ARG, "crf is NULL");
    LCCRF_TRY(lccrf_crf_start(crf));
    for (int it = 0; it < n_iterations; it++) LCCRF_TRY(lccrf_crf_step(crf, relax));
    if (with_map) LCCRF_TRY(lccrf_crf_build_map(crf));
    // results must be host-visible when inference() returns (Tracking.cc:1930-1948 indexes them directly)
    return crf_fetch(crf);
}

const short *lccrf_crf_map(lccrf_crf *crf) {
    if (!crf || !crf->map_built) return nullptr;
    cudaSetDevice(crf->ctx->device);
    if (crf_fetch(crf) != LCCRF_OK) return nullptr;
    return crf->h_map;
}

const float *lccrf_crf_prob(lccrf_crf *crf) {
    if (!crf) return nullptr;
    cudaSetDevice(crf->ctx->device);
    if (!crf->started) {
        // current_ exists from construction in the reference (uninitialised); hand out the buffer
        return crf->h_prob;
    }
    if (crf_fetch(crf) != LCCRF_OK) return nullptr;
    return crf->h_prob;
}

int lccrf_crf_potts_vertices(const lccrf_crf *crf, int k, int *V) {
    if (!crf || !V) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (k < 0 || k >= (int)crf->b.lat.size()) return fail(LCCRF_ERR_ARG, "potential index out of range");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    LCCRF_CUDA(cudaMemcpyAsync(ctx->h_status, crf->b.lat[k]->vbase + 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    *V = *ctx->h_status;
    return LCCRF_OK;
}

int lccrf_crf_num_potts(const lccrf_crf *crf) { return crf ? (int)crf->b.lat.size() : 0; }

int lccrf_crf_step_init(lccrf_crf *crf, float *next) {
    if (!crf || !next) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)crf->b.NT * crf->b.L;
    if (!n) return LCCRF_OK;
    LCCRF_TRY(mf_negate(ctx, crf->b.next, crf->b.unary, (long long)n));
    LCCRF_CUDA(cudaMemcpyAsync(next, crf->b.next, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

int lccrf_crf_set_prob(lccrf_crf *crf, const float *prob) {
    if (!crf || !prob) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)crf->b.NT * crf->b.L;
    if (n) LCCRF_CUDA(cudaMemcpyAsync(crf->b.cur, prob, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    crf->started = true;
    crf->prob_fresh = false;
    return LCCRF_OK;
}

int lccrf_crf_potts_apply(lccrf_crf *crf, int k, float *out, const float *in, float *tmp) {
    if (!crf || !out || !in || !tmp) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (k < 0 || k >= (int)crf->b.lat.size()) return fail(LCCRF_ERR_ARG, "potential index out of range");
    Ctx *ctx = crf->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)crf->b.NT * crf->b.L;
    if (!n) return LCCRF_OK;
    // device staging: next <- out, cur-like scratch <- in (b.tmp holds `in`, dev_io holds tmp)
    LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, 3 * n * sizeof(float)));
    float *d_out = (float *)ctx->dev_io.p, *d_in = d_out + n, *d_tmp = d_in + n;
    LCCRF_CUDA(cudaMemcpyAsync(d_out, out, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaMemcpyAsync(d_in, in, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_TRY(mf_potts_apply(ctx, crf->b, crf->b.lat[k], d_out, d_in, d_tmp, crf->b.L));
    LCCRF_CUDA(cudaMemcpyAsync(out, d_out, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaMemcpyAsync(tmp, d_tmp, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

int lccrf_exp_and_normalize(lccrf_ctx *h, float *out, const float *in, int N, int L, float scale, float relax) {
    if (!h || !out || !in) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (N < 0 || L < 1 || L > LCCRF_MAX_L) return fail(LCCRF_ERR_ARG, "N or L out of range");
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)N * L;
    if (!n) return LCCRF_OK;
    LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, 2 * n * sizeof(float)));
    float *d_out = (float *)ctx->dev_io.p, *d_in = d_out + n;
    LCCRF_CUDA(cudaMemcpyAsync(d_in, in, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if (relax != 1.0f) LCCRF_CUDA(cudaMemcpyAsync(d_out, out, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_TRY(mf_exp_and_normalize(ctx, d_out, d_in, N, L, scale, relax));
    LCCRF_CUDA(cudaMemcpyAsync(out, d_out, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

// ------------------------------------------------------------------ long-term unary (host-pointer calls)
int lccrf_map_point_unary(lccrf_ctx *h, int N, const float *xyz, const int *obs_ptr, const int *obs_kf,
                          const float *obs_uv, int nKF, const float *kf_pose, const float *kf_intr,
                          const float *kf_bounds, float *observs, float *error, float *depth) {
    if (!h) return fail(LCCRF_ERR_ARG, "ctx is NULL");
    if (N < 0 || nKF < 0) return fail(LCCRF_ERR_ARG, "negative size");
    if (N == 0) return LCCRF_OK;
    if (!xyz || !obs_ptr || !observs || !error || !depth) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const long long nnz = obs_ptr[N];
    if (obs_ptr[0] != 0 || nnz < 0) return fail(LCCRF_ERR_ARG, "obs_ptr must start at 0");
    for (int i = 0; i < N; i++)
        if (obs_ptr[i + 1] < obs_ptr[i]) return fail(LCCRF_ERR_ARG, "obs_ptr must be non-decreasing");
    if (nnz > 0 && (!obs_kf || !obs_uv || !kf_pose || !kf_intr || !kf_bounds)) return fail(LCCRF_ERR_ARG, "NULL argument");
    for (long long e = 0; e < nnz; e++)
        if (obs_kf[e] < 0 || obs_kf[e] >= nKF) return fail(LCCRF_ERR_ARG, "obs_kf out of range");
    // device staging
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t o_xyz = take((size_t)N * 12), o_ptr = take((size_t)(N + 1) * 4), o_kf = take((size_t)nnz * 4),
                 o_uv = take((size_t)nnz * 8), o_pose = take((size_t)nKF * 48), o_intr = take((size_t)nKF * 16),
                 o_bnd = take((size_t)nKF * 16), o_out = take((size_t)N * 12);
    LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, off + 256));
    char *base = (char *)ctx->dev_io.p;
    cudaStream_t st = ctx->stream;
    LCCRF_CUDA(cudaMemcpyAsync(base + o_xyz, xyz, (size_t)N * 12, cudaMemcpyHostToDevice, st));
    LCCRF_CUDA(cudaMemcpyAsync(base + o_ptr, obs_ptr, (size_t)(N + 1) * 4, cudaMemcpyHostToDevice, st));
    if (nnz) {
        LCCRF_CUDA(cudaMemcpyAsync(base + o_kf, obs_kf, (size_t)nnz * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(base + o_uv, obs_uv, (size_t)nnz * 8, cudaMemcpyHostToDevice, st));
    }
    if (nKF) {
        LCCRF_CUDA(cudaMemcpyAsync(base + o_pose, kf_pose, (size_t)nKF * 48, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(base + o_intr, kf_intr, (size_t)nKF * 16, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(base + o_bnd, kf_bounds, (size_t)nKF * 16, cudaMemcpyHostToDevice, st));
    }
    float *d_obs = (float *)(base + o_out), *d_err = d_obs + N, *d_dep = d_err + N;
    float cam8[8];
    const bool ucam = uniform_camera(kf_intr, kf_bounds, nKF, cam8);
    LCCRF_TRY(unary_map_points(ctx, N, (const float *)(base + o_xyz), (const int *)(base + o_ptr),
                               (const int *)(base + o_kf), (const float *)(base + o_uv), nKF,
                               (const float *)(base + o_pose), (const float *)(base + o_intr),
                               (const float *)(base + o_bnd), d_obs, d_err, d_dep, ucam ? cam8 : nullptr));
    LCCRF_CUDA(cudaMemcpyAsync(observs, d_obs, (size_t)N * 4, cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaMemcpyAsync(error, d_err, (size_t)N * 4, cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaMemcpyAsync(depth, d_dep, (size_t)N * 4, cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));
    return LCCRF_OK;
}

int lccrf_rough_classify(lccrf_ctx *h, int N, const float *observs, const float *error, const float *depth,
                         const double *p4, const lccrf_slam_params *prm, short *label) {
    if (!h || !prm) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (N < 0) return fail(LCCRF_ERR_ARG, "N < 0");
    if (N == 0) return LCCRF_OK;
    if (!observs || !error || !depth || !label) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n4 = ((size_t)N * 4 + 255) / 256 * 256;
    LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, 3 * n4 + (size_t)N * 8 + 256 + (size_t)N * 2 + 256));
    char *base = (char *)ctx->dev_io.p;
    float *d_o = (float *)base, *d_e = (float *)(base + n4), *d_d = (float *)(base + 2 * n4);
    double *d_p4 = (double *)(base + 3 * n4);
    short *d_lab = (short *)(base + 3 * n4 + ((size_t)N * 8 + 255) / 256 * 256);
    cudaStream_t st = ctx->stream;
    LCCRF_CUDA(cudaMemcpyAsync(d_o, observs, (size_t)N * 4, cudaMemcpyHostToDevice, st));
    LCCRF_CUDA(cudaMemcpyAsync(d_e, error, (size_t)N * 4, cudaMemcpyHostToDevice, st));
    LCCRF_CUDA(cudaMemcpyAsync(d_d, depth, (size_t)N * 4, cudaMemcpyHostToDevice, st));
    if (p4) LCCRF_CUDA(cudaMemcpyAsync(d_p4, p4, (size_t)N * 8, cudaMemcpyHostToDevice, st));
    LCCRF_TRY(unary_classify(ctx, N, d_o, d_e, d_d, p4 ? d_p4 : nullptr, *prm, d_lab));
    LCCRF_CUDA(cudaMemcpyAsync(label, d_lab, (size_t)N * 2, cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));
    return LCCRF_OK;
}

// ------------------------------------------------------------------ frontend: epipolar prior, BfMatch
int lccrf_epipolar_prior(lccrf_ctx *h, int M, const int *fid1, const float *pt1, const float *pt2, const double *F9,
                         float u_gamma, float stdev_gamma, int nFeat, double *dis_by_fid, double *prob_by_fid,
                         double *dis, double *prob) {
    if (!h) return fail(LCCRF_ERR_ARG, "ctx is NULL");
    if (M < 0 || nFeat < 0) return fail(LCCRF_ERR_ARG, "negative size");
    if ((dis_by_fid || prob_by_fid) && !fid1 && M > 0) return fail(LCCRF_ERR_ARG, "fid1 is required for the by-feature outputs");
    if (M > 0 && (!pt1 || !pt2 || !F9)) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (fid1)
        for (int m = 0; m < M; m++)
            if (fid1[m] < 0 || fid1[m] >= nFeat) return fail(LCCRF_ERR_ARG, "fid1 out of range");
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t o_fid = take((size_t)M * 4), o_p1 = take((size_t)M * 8), o_p2 = take((size_t)M * 8),
                 o_dm = take((size_t)M * 8), o_pm = take((size_t)M * 8), o_df = take((size_t)nFeat * 8),
                 o_pf = take((size_t)nFeat * 8);
    LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, off + 256));
    char *base = (char *)ctx->dev_io.p;
    cudaStream_t st = ctx->stream;
    if (M > 0) {
        if (fid1) LCCRF_CUDA(cudaMemcpyAsync(base + o_fid, fid1, (size_t)M * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(base + o_p1, pt1, (size_t)M * 8, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(base + o_p2, pt2, (size_t)M * 8, cudaMemcpyHostToDevice, st));
    }
    // unmatched features read 0.0, the value std::map<int,double>::operator[] inserts (Tracking.cc:2003)
    if (nFeat > 0) LCCRF_CUDA(cudaMemsetAsync(base + o_df, 0, (o_pf - o_df) + (size_t)nFeat * 8, st));
    LCCRF_TRY(epipolar_prior(ctx, M, fid1 ? (const int *)(base + o_fid) : nullptr, (const float *)(base + o_p1),
                             (const float *)(base + o_p2), F9, u_gamma, stdev_gamma, nFeat,
                             dis_by_fid ? (double *)(base + o_df) : nullptr, prob_by_fid ? (double *)(base + o_pf) : nullptr,
                             (double *)(base + o_dm), (double *)(base + o_pm)));
    if (dis && M > 0) LCCRF_CUDA(cudaMemcpyAsync(dis, base + o_dm, (size_t)M * 8, cudaMemcpyDeviceToHost, st));
    if (prob && M > 0) LCCRF_CUDA(cudaMemcpyAsync(prob, base + o_pm, (size_t)M * 8, cudaMemcpyDeviceToHost, st));
    if (dis_by_fid && nFeat > 0) LCCRF_CUDA(cudaMemcpyAsync(dis_by_fid, base + o_df, (size_t)nFeat * 8, cudaMemcpyDeviceToHost, st));
    if (prob_by_fid && nFeat > 0) LCCRF_CUDA(cudaMemcpyAsync(prob_by_fid, base + o_pf, (size_t)nFeat * 8, cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));
    return LCCRF_OK;
}

int lccrf_bf_match_batch(lccrf_ctx *h, int B, const int *q_ptr, const uint8_t *desc_q, const int *t_ptr,
                         const uint8_t *desc_t, double ratio, int *match, int *knn, int *n_match) {
    if (!h) return fail(LCCRF_ERR_ARG, "ctx is NULL");
    if (B < 0 || B > 65535) return fail(LCCRF_ERR_ARG, "B must be in [0, 65535]");
    if (n_match) *n_match = 0;
    if (B == 0) return LCCRF_OK;
    if (!q_ptr || !t_ptr) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (q_ptr[0] != 0 || t_ptr[0] != 0) return fail(LCCRF_ERR_ARG, "q_ptr / t_ptr must start at 0");
    int max_nq = 0, max_nt = 0;
    for (int b = 0; b < B; b++) {
        const int nq = q_ptr[b + 1] - q_ptr[b], nt = t_ptr[b + 1] - t_ptr[b];
        if (nq < 0 || nt < 0) return fail(LCCRF_ERR_ARG, "q_ptr / t_ptr must be non-decreasing");
        if (nq > max_nq) max_nq = nq;
        if (nt > max_nt) max_nt = nt;
    }
    const int NQ = q_ptr[B], NTr = t_ptr[B];
    if (NQ == 0) return LCCRF_OK;
    if (!desc_q || (NTr > 0 && !desc_t) || !match) return fail(LCCRF_ERR_ARG, "NULL argument");
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const int S = bf_match_splits(B, max_nq, max_nt);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t o_qp = take((size_t)(B + 1) * 4), o_tp = take((size_t)(B + 1) * 4), o_dq = take((size_t)NQ * 32),
                 o_dt = take((size_t)NTr * 32), o_part = take((size_t)NQ * S * 16), o_match = take((size_t)NQ * 4),
                 o_knn = take((size_t)NQ * 16), o_cnt = take(4);
    LCCRF_TRY(ctx_scratch(ctx, ctx->dev_io, off + 256));
    char *base = (char *)ctx->dev_io.p;
    cudaStream_t st = ctx->stream;
    LCCRF_CUDA(cudaMemcpyAsync(base + o_qp, q_ptr, (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, st));
    LCCRF_CUDA(cudaMemcpyAsync(base + o_tp, t_ptr, (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, st));
    LCCRF_CUDA(cudaMemcpyAsync(base + o_dq, desc_q, (size_t)NQ * 32, cudaMemcpyHostToDevice, st));
    if (NTr > 0) LCCRF_CUDA(cudaMemcpyAsync(base + o_dt, desc_t, (size_t)NTr * 32, cudaMemcpyHostToDevice, st));
    LCCRF_TRY(bf_match(ctx, B, NQ, max_nq, max_nt, (const int *)(base + o_qp), base + o_dq, (const int *)(base + o_tp),
                       base + o_dt, ratio, S, base + o_part, (int *)(base + o_match), knn ? (int *)(base + o_knn) : nullptr,
                       (int *)(base + o_cnt)));
    LCCRF_CUDA(cudaMemcpyAsync(match, base + o_match, (size_t)NQ * 4, cudaMemcpyDeviceToHost, st));
    if (knn) LCCRF_CUDA(cudaMemcpyAsync(knn, base + o_knn, (size_t)NQ * 16, cudaMemcpyDeviceToHost, st));
    int cnt = 0;
    LCCRF_CUDA(cudaMemcpyAsync(&cnt, base + o_cnt, 4, cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));
    if (n_match) *n_match = cnt;
    return LCCRF_OK;
}

int lccrf_bf_match(lccrf_ctx *h, int nq, const uint8_t *desc_q, int nt, const uint8_t *desc_t, double ratio, int *match,
                   int *knn, int *n_match) {
    if (nq < 0 || nt < 0) return fail(LCCRF_ERR_ARG, "negative size");
    const int qp[2] = {0, nq}, tp[2] = {0, nt};
    return lccrf_bf_match_batch(h, 1, qp, desc_q, tp, desc_t, ratio, match, knn, n_match);
}

// ------------------------------------------------------------------ device-resident map
int lccrf_map_create(lccrf_ctx *h, int kp_stride, lccrf_map **out) {
    if (!h || !out) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (kp_stride < 1 || kp_stride > (1 << 20)) return fail(LCCRF_ERR_ARG, "kp_stride must be in [1, 2^20]");
    *out = nullptr;
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    auto *mp = new lccrf_map();
    int rc = map_create(ctx, kp_stride, &mp->m);
    if (rc != LCCRF_OK) {
        delete mp;
        return rc;
    }
    *out = mp;
    return LCCRF_OK;
}

void lccrf_map_destroy(lccrf_map *map) {
    if (!map) return;
    if (map->m) {
        cudaSetDevice(map->m->ctx->device);
        map_destroy(map->m);
    }
    delete map;
}

int lccrf_map_apply(lccrf_map *map, const lccrf_map_delta *delta) {
    if (!map || !map->m || !delta) return fail(LCCRF_ERR_ARG, "NULL argument");
    DevMap *m = map->m;
    Ctx *ctx = m->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    LCCRF_TRY(map_begin_main_access(m));  // behind the asynchronous mutations of earlier pipelined submissions
    LCCRF_TRY(map_prepare(m, *delta));
    LCCRF_TRY(delta_grow_points(m, *delta));
    void *stage = nullptr;
    LCCRF_TRY(dev_alloc(ctx, &stage, delta_stage_bytes(*delta, m->kp_stride, false)));
    DeltaDev dd;
    int rc = delta_stage(*delta, m->kp_stride, false, (char *)stage, ctx->stream, &dd);
    if (rc == LCCRF_OK) rc = map_apply_dev(m, dd, delta->kf_count > 0 ? delta->kf_keypoints : nullptr);
    dev_free(ctx, stage);
    if (rc != LCCRF_OK) return rc;
    return check_status(ctx);  // synchronises: the host arrays are free on return
}

int lccrf_map_set_observations(lccrf_map *map, int pt_first, int count, const int *obs_ptr, const int *obs_ref) {
    if (!map || !map->m) return fail(LCCRF_ERR_ARG, "map is NULL");
    if (pt_first < 0 || count < 0) return fail(LCCRF_ERR_ARG, "negative point range");
    if (count == 0) return LCCRF_OK;
    if (!obs_ptr) return fail(LCCRF_ERR_ARG, "obs_ptr is NULL");
    DevMap *m = map->m;
    Ctx *ctx = m->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    if (obs_ptr[0] != 0) return fail(LCCRF_ERR_ARG, "obs_ptr must start at 0");
    const long long nnz = obs_ptr[count];
    if (nnz > 0 && !obs_ref) return fail(LCCRF_ERR_ARG, "obs_ref is NULL");
    // tight runs by default; option "map_slack" (percent, at least 2 entries when set) leaves room so that the first appends
    // do not move the list
    std::vector<int> ptrs(2 * (size_t)count + 2);
    long long run = 0;
    for (int i = 0; i < count; i++) {
        const int c = obs_ptr[i + 1] - obs_ptr[i];
        if (c < 0) return fail(LCCRF_ERR_ARG, "obs_ptr must be non-decreasing");
        ptrs[i] = obs_ptr[i];
        ptrs[count + 1 + i] = (int)run;
        const int extra = (int)(((long long)c * ctx->opt_map_slack + 99) / 100);
        run += c + (ctx->opt_map_slack > 0 && extra < 2 ? 2 : extra);
        if (run > 0x7fffffffLL) return fail(LCCRF_ERR_ARG, "bulk load exceeds 2^31 pool entries");
    }
    ptrs[count] = (int)nnz;
    ptrs[2 * (size_t)count + 1] = (int)run;
    if ((long long)pt_first + count > 0x7fffffffLL) return fail(LCCRF_ERR_ARG, "point id overflow");
    LCCRF_TRY(map_begin_main_access(m));
    LCCRF_TRY(map_reserve_points(m, pt_first + count));
    if (pt_first + count > m->n_pt) m->n_pt = pt_first + count;
    LCCRF_TRY(map_bulk_reserve(m, run));
    int *d_ptrs = nullptr, *d_ref = nullptr;
    LCCRF_TRY(dev_alloc(ctx, (void **)&d_ptrs, ptrs.size() * 4));
    int rc = dev_alloc(ctx, (void **)&d_ref, (size_t)(nnz > 0 ? nnz : 1) * 8);
    if (rc == LCCRF_OK) {
        cudaError_t e = cudaMemcpyAsync(d_ptrs, ptrs.data(), ptrs.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess && nnz > 0) e = cudaMemcpyAsync(d_ref, obs_ref, (size_t)nnz * 8, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
    }
    if (rc == LCCRF_OK) rc = map_bulk_observations(m, pt_first, count, d_ptrs, d_ref, nnz, 25);
    dev_free(ctx, d_ptrs);
    dev_free(ctx, d_ref);
    if (rc != LCCRF_OK) return rc;
    rc = check_status(ctx);  // synchronises
    map_counters(m, nullptr, nullptr);
    return rc;
}

int lccrf_map_reserve_observations(lccrf_map *map, long long entries) {
    if (!map || !map->m) return fail(LCCRF_ERR_ARG, "map is NULL");
    if (entries < 0) return fail(LCCRF_ERR_ARG, "negative size");
    DevMap *m = map->m;
    LCCRF_CUDA(cudaSetDevice(m->ctx->device));
    long long tail = 0;
    LCCRF_TRY(map_counters(m, &tail, nullptr));
    return map_reserve_pool(m, tail + entries);
}

int lccrf_map_sizes(lccrf_map *map, int *n_kf, int *n_points, long long *n_obs, long long *pool_used, long long *pool_cap) {
    if (!map || !map->m) return fail(LCCRF_ERR_ARG, "map is NULL");
    DevMap *m = map->m;
    LCCRF_CUDA(cudaSetDevice(m->ctx->device));
    long long tail = 0, live = 0;
    LCCRF_TRY(map_counters(m, &tail, &live));
    if (n_kf) *n_kf = m->n_kf;
    if (n_points) *n_points = m->n_pt;
    if (n_obs) *n_obs = live;
    if (pool_used) *pool_used = tail;
    if (pool_cap) *pool_cap = m->pool_cap;
    return LCCRF_OK;
}

int lccrf_map_export(lccrf_map *map, int n, const int *point_id, int *obs_ptr, int *obs_kf, float *obs_uv, long long cap,
                     float *xyz) {
    if (!map || !map->m) return fail(LCCRF_ERR_ARG, "map is NULL");
    if (n < 0 || cap < 0) return fail(LCCRF_ERR_ARG, "negative size");
    if (n == 0) return LCCRF_OK;
    if (!point_id || !obs_ptr) return fail(LCCRF_ERR_ARG, "NULL argument");
    DevMap *m = map->m;
    Ctx *ctx = m->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    int *d_ids = nullptr, *d_ptr = nullptr;
    LCCRF_TRY(dev_alloc(ctx, (void **)&d_ids, (size_t)n * 4));
    int rc = dev_alloc(ctx, (void **)&d_ptr, ((size_t)n + 1) * 4);
    std::vector<int> cnt((size_t)n + 1);
    if (rc == LCCRF_OK) {
        cudaError_t e = cudaMemcpyAsync(d_ids, point_id, (size_t)n * 4, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
    }
    if (rc == LCCRF_OK) rc = map_export_dev(m, n, d_ids, d_ptr);
    if (rc == LCCRF_OK) {
        cudaError_t e = cudaMemcpyAsync(cnt.data(), d_ptr, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
    }
    long long tot = 0;
    if (rc == LCCRF_OK) {
        for (int i = 0; i < n; i++) {
            obs_ptr[i] = (int)tot;
            tot += cnt[i];
        }
        obs_ptr[n] = (int)tot;
        if (tot > cap && (obs_kf || obs_uv)) rc = fail(LCCRF_ERR_ARG, "lccrf_map_export: output capacity too small (obs_ptr[n] tells the need)");
    }
    int *d_kf = nullptr;
    float *d_uv = nullptr, *d_xyz = nullptr;
    if (rc == LCCRF_OK && (obs_kf || obs_uv || xyz)) {
        const size_t ne = (size_t)(tot > 0 ? tot : 1);
        rc = dev_alloc(ctx, (void **)&d_kf, ne * 4);
        if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&d_uv, ne * 8);
        if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&d_xyz, (size_t)n * 12);
        if (rc == LCCRF_OK) {
            cudaError_t e = cudaMemcpyAsync(d_ptr, obs_ptr, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
        }
        if (rc == LCCRF_OK) rc = map_export_entries_dev(m, n, d_ids, d_ptr, d_kf, d_uv, d_xyz, tot);
        if (rc == LCCRF_OK) {
            cudaError_t e = cudaSuccess;
            if (obs_kf && tot) e = cudaMemcpyAsync(obs_kf, d_kf, (size_t)tot * 4, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess && obs_uv && tot) e = cudaMemcpyAsync(obs_uv, d_uv, (size_t)tot * 8, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess && xyz) e = cudaMemcpyAsync(xyz, d_xyz, (size_t)n * 12, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
        }
    }
    dev_free(ctx, d_ids);
    dev_free(ctx, d_ptr);
    dev_free(ctx, d_kf);
    dev_free(ctx, d_uv);
    dev_free(ctx, d_xyz);
    if (rc != LCCRF_OK) return rc;
    return check_status(ctx);
}

}  // extern "C"
