// api.cu -- the extern "C" boundary (include/lccrf.h) and the host-side engine objects.
#include <chrono>
#include <climits>
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
static int decode_status(int st) {
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

// host-side phase timer of the pipelined submit path (option "trace": one line per submission on stderr)
struct PhaseTimer {
    bool on;
    std::chrono::steady_clock::time_point t0;
    std::string line;
    explicit PhaseTimer(bool enable) : on(enable), t0(std::chrono::steady_clock::now()) {}
    void mark(const char *what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        char buf[64];
        snprintf(buf, sizeof(buf), " %s=%.0fus", what, std::chrono::duration<double, std::micro>(t1 - t0).count());
        line += buf;
        t0 = t1;
    }
    ~PhaseTimer() {
        if (on) fprintf(stderr, "lccrf trace:%s\n", line.c_str());
    }
};

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

struct lccrf_map {
    DevMap *m = nullptr;
};

// one set of device-resident inputs of a frames batch.  Two sets exist so that lccrf_frames_submit_* can upload
// step i+1 on the copy stream while step i computes (the graph of a slot reads that slot's buffers).
struct FrameInputs {
    // direct inputs (Tracking.cc:1849-1870 vectors) -- used when !from_map
    float *observs = nullptr, *error = nullptr, *depth = nullptr;
    float *kp2d = nullptr;  // [NT*2], both modes
    // map snapshot
    bool from_map = false;
    float *xyz = nullptr, *obs_uv = nullptr, *kf_pose = nullptr, *kf_intr = nullptr, *kf_bounds = nullptr;
    int *obs_ptr = nullptr;
    void *obs_kf = nullptr;  // int32 or uint16 keyframe indices
    int obs_kf_bytes = 4;
    void *kf_packed = nullptr;
    int *kf_ptr = nullptr;  // [B+1] keyframe slice of each problem (optional)
    bool have_kf_ptr = false;
    int nKF = 0, nKF_cap = 0;
    int kf_slice_max = 0;  // largest per-problem keyframe slice (0 = unknown)
    bool ucam = false;     // every keyframe has the same intrinsics / image bounds (cam8)
    float cam8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long nnz = 0, nnz_cap = 0;
    bool indexed = false;  // obs_kf holds {keyframe, feature index} pairs; keypoints come from lccrf_frames::kp_tab
    // frame points named by ids of a device-resident map (lccrf_frames_set_visible / submit_visible)
    bool visible = false;
    DevMap *map = nullptr;
    int *vis = nullptr;       // [NT] map point ids
    uint64_t map_gen = 0;
    int kf_bucket = 0;        // shared-memory keyframe slots the captured graph was sized for
    void *out_stage = nullptr;     // per-slot copy of the results (marginals, labels, status word) on their way to the host
    cudaEvent_t res_ready = nullptr;
    void *stage = nullptr;    // staged arrays of this step's map delta
    size_t stage_cap = 0;
    DeltaDev delta;
    bool has_delta = false;
    // epipolar prior (lccrf_frames_set_prior): host arrays as registered, device copies
    const double *h_p4 = nullptr;
    const unsigned char *h_p4_has = nullptr;
    double *p4 = nullptr;
    unsigned char *p4_has = nullptr;
    bool use_p4 = false, use_p4_has = false;
    // label-application lists delivered by the pipelined submissions (lccrf_frames_set_partition_outputs)
    const int *part_fid = nullptr;
    int *part_dyn_ptr = nullptr, *part_dyn = nullptr, *part_stat_ptr = nullptr, *part_stat = nullptr;
    bool have_inputs = false;
    GraphReplay graph;
    uint64_t kp_gen = 0;
    cudaEvent_t up_done = nullptr, run_done = nullptr, out_done = nullptr;
    int *h_status = nullptr;  // pinned copy of the device status word taken after this slot's run
    bool in_flight = false;
};

struct lccrf_frames {
    Ctx *ctx = nullptr;
    Batch b;
    lccrf_slam_params prm;
    float energies[3];
    float *d_en = nullptr;  // n_en[2], p_en[2]
    float *observs = nullptr, *error = nullptr, *depth = nullptr;  // device [NT]: outputs of the unary kernel
    short *label = nullptr;
    float *feat = nullptr, *feat2 = nullptr;  // [NT*2] features of the appearance / smoothness kernel
    FrameInputs in[2];
    int last_slot = 0;
    bool ran = false;
    int *part = nullptr;  // label application workspace: dyn_ptr, stat_ptr [B+1], dyn_list, stat_list, fid [NT], tiles
    // resident keyframe keypoints (KeyFrame::mvKeysUn, immutable per keyframe): [kp_cap][kp_stride] float2
    float *kp_tab = nullptr;
    int kp_cap = 0, kp_stride = 0;
    uint64_t kp_gen = 0;  // bumped when the table moves (captured graphs hold its address)
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
        scratch_release(c, bs.blk_cnt, false);
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

int lccrf_ctx_set_option(lccrf_ctx *h, const char *name, int value) {
    if (!h || !name) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (!strcmp(name, "graphs")) h->c.opt_graphs = value;
    else if (!strcmp(name, "fused")) h->c.opt_fused = value;
    else if (!strcmp(name, "ordered_splat")) {
        if (h->c.opt_ordered_splat != (value ? 1 : 0)) h->c.scratch_gen++;  // captured graphs hold the other kernel set
        h->c.opt_ordered_splat = value ? 1 : 0;
    }
    else if (!strcmp(name, "profile")) h->c.opt_profile = value;
    else if (!strcmp(name, "map_slack")) h->c.opt_map_slack = value < 0 ? 0 : value;
    else if (!strcmp(name, "trace")) h->c.opt_trace = value;
    else if (!strcmp(name, "bulk_blur")) {
        if (h->c.opt_bulk_blur != (value ? 1 : 0)) h->c.scratch_gen++;
        h->c.opt_bulk_blur = value ? 1 : 0;
    }
    else if (!strcmp(name, "concurrent")) {
        if (h->c.opt_concurrent != value) h->c.scratch_gen++;  // captured graphs hold the other branch structure
        h->c.opt_concurrent = value;
    }
    else if (!strcmp(name, "split_splat")) {
        if (h->c.opt_split_splat != (value ? 1 : 0)) h->c.scratch_gen++;
        h->c.opt_split_splat = value ? 1 : 0;
    }
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

// ------------------------------------------------------------------ batched frames
int lccrf_frames_create(lccrf_ctx *h, int B, const int *prob_ptr, const lccrf_slam_params *prm,
                        const float *energies3, lccrf_frames **out) {
    if (!h || !out || !prob_ptr || !prm || !energies3) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (B < 1) return fail(LCCRF_ERR_ARG, "B must be >= 1");
    if (prm->iters < 0) return fail(LCCRF_ERR_ARG, "iters < 0");
    *out = nullptr;
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    auto *fr = new lccrf_frames();
    fr->ctx = ctx;
    fr->prm = *prm;
    memcpy(fr->energies, energies3, sizeof(fr->energies));
    int rc = batch_init(ctx, fr->b, B, prob_ptr, 2, true);
    const size_t n = (size_t)(fr->b.NT > 0 ? fr->b.NT : 1);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&fr->observs, n * 4);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&fr->error, n * 4);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&fr->depth, n * 4);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&fr->feat, n * 8);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&fr->feat2, n * 8);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&fr->label, n * 2);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&fr->d_en, 4 * sizeof(float));
    if (rc == LCCRF_OK) {
        float en[4] = {energies3[1], energies3[1], energies3[2], energies3[2]};  // n_en[2], p_en[2]
        cudaError_t e = cudaMemcpyAsync(fr->d_en, en, sizeof(en), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
    }
    for (int k = 0; k < 2 && rc == LCCRF_OK; k++) {
        LatticeSet *ls = nullptr;
        rc = lattice_set_create(ctx, fr->b, 2, k == 0 ? prm->w1 : prm->w2, 2, &ls);
        if (rc == LCCRF_OK) fr->b.lat.push_back(ls);
    }
    if (rc != LCCRF_OK) {
        lccrf_frames_destroy(fr);
        return rc;
    }
    *out = fr;
    return LCCRF_OK;
}

static void frame_inputs_release(Ctx *ctx, FrameInputs &in) {
    graph_drop(in.graph);
    dev_free(ctx, in.observs);
    dev_free(ctx, in.error);
    dev_free(ctx, in.depth);
    dev_free(ctx, in.kp2d);
    dev_free(ctx, in.xyz);
    dev_free(ctx, in.obs_uv);
    dev_free(ctx, in.kf_pose);
    dev_free(ctx, in.kf_intr);
    dev_free(ctx, in.kf_bounds);
    dev_free(ctx, in.obs_ptr);
    dev_free(ctx, in.obs_kf);
    dev_free(ctx, in.kf_packed);
    dev_free(ctx, in.kf_ptr);
    dev_free(ctx, in.vis);
    dev_free(ctx, in.out_stage);
    if (in.res_ready) cudaEventDestroy(in.res_ready);
    dev_free(ctx, in.p4);
    dev_free(ctx, in.p4_has);
    if (in.stage) cudaFree(in.stage);
    if (in.up_done) cudaEventDestroy(in.up_done);
    if (in.run_done) cudaEventDestroy(in.run_done);
    if (in.out_done) cudaEventDestroy(in.out_done);
    if (in.h_status) cudaFreeHost(in.h_status);
    in = FrameInputs();
}

void lccrf_frames_destroy(lccrf_frames *fr) {
    if (!fr) return;
    Ctx *ctx = fr->ctx;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->d2h_stream) cudaStreamSynchronize(ctx->d2h_stream);
    for (auto &in : fr->in) frame_inputs_release(ctx, in);
    batch_release(ctx, fr->b);
    dev_free(ctx, fr->observs);
    dev_free(ctx, fr->error);
    dev_free(ctx, fr->depth);
    dev_free(ctx, fr->feat);
    dev_free(ctx, fr->feat2);
    dev_free(ctx, fr->label);
    dev_free(ctx, fr->d_en);
    dev_free(ctx, fr->part);
    dev_free(ctx, fr->kp_tab);
    delete fr;
}

// upload the direct per-frame vectors of one step into input set `in` on stream `st`
// Input buffers are stream-ordered allocations of ctx->stream, but the pipelined submit path fills them on the copy
// stream: after a (re)allocation the copy stream is ordered behind ctx->stream once, so that a block the pool recycled
// from work still running there (the other slot's step) is not overwritten early.  Steady state allocates nothing.
static int order_copies_after_alloc(Ctx *ctx, FrameInputs &in, cudaStream_t st) {
    if (st == ctx->stream || !in.up_done) return LCCRF_OK;
    LCCRF_CUDA(cudaEventRecord(in.up_done, ctx->stream));
    LCCRF_CUDA(cudaStreamWaitEvent(st, in.up_done, 0));
    return LCCRF_OK;
}

// epipolar prior registered with lccrf_frames_set_prior: uploaded with the slot's other inputs
static int frames_upload_prior(lccrf_frames *fr, FrameInputs &in, cudaStream_t st) {
    Ctx *ctx = fr->ctx;
    const bool use = in.h_p4 != nullptr && fr->b.NT > 0, use_has = use && in.h_p4_has != nullptr;
    if (use != in.use_p4 || use_has != in.use_p4_has) graph_drop(in.graph);  // the classifier's arguments change
    in.use_p4 = use;
    in.use_p4_has = use_has;
    if (!use) return LCCRF_OK;
    bool fresh = false;
    if (!in.p4) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.p4, (size_t)fr->b.NT * sizeof(double)));
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.p4_has, (size_t)fr->b.B));
        graph_drop(in.graph);
        fresh = true;
    }
    if (fresh) LCCRF_TRY(order_copies_after_alloc(ctx, in, st));
    LCCRF_CUDA(cudaMemcpyAsync(in.p4, in.h_p4, (size_t)fr->b.NT * sizeof(double), cudaMemcpyHostToDevice, st));
    if (use_has) LCCRF_CUDA(cudaMemcpyAsync(in.p4_has, in.h_p4_has, (size_t)fr->b.B, cudaMemcpyHostToDevice, st));
    return LCCRF_OK;
}

static int frames_upload_direct(lccrf_frames *fr, FrameInputs &in, cudaStream_t st, const float *observs,
                                const float *error, const float *depth, const float *kp2d) {
    Ctx *ctx = fr->ctx;
    const size_t n = (size_t)fr->b.NT;
    if (n && (!observs || !error || !depth || !kp2d)) return fail(LCCRF_ERR_ARG, "NULL argument");
    bool fresh = false;
    if (!in.observs) {
        const size_t m = n ? n : 1;
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.observs, m * 4));
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.error, m * 4));
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.depth, m * 4));
        graph_drop(in.graph);
        fresh = true;
    }
    if (!in.kp2d) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kp2d, (n ? n : 1) * 8));
        graph_drop(in.graph);
        fresh = true;
    }
    if (fresh) LCCRF_TRY(order_copies_after_alloc(ctx, in, st));
    if (in.from_map) graph_drop(in.graph);
    in.from_map = false;
    in.visible = false;
    LCCRF_TRY(frames_upload_prior(fr, in, st));
    if (n) {
        LCCRF_CUDA(cudaMemcpyAsync(in.observs, observs, n * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.error, error, n * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.depth, depth, n * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kp2d, kp2d, n * 8, cudaMemcpyHostToDevice, st));
    }
    in.have_inputs = true;
    return LCCRF_OK;
}

// validate + upload a map snapshot of one step into input set `in` on stream `st`
static int frames_upload_map(lccrf_frames *fr, FrameInputs &in, cudaStream_t st, const float *xyz, const int *obs_ptr,
                             const void *obs_kf, int obs_kf_bytes, const float *obs_uv, int nKF, const float *kf_pose,
                             const float *kf_intr, const float *kf_bounds, const float *kp2d, const int *kf_ptr,
                             bool indexed = false) {
    Ctx *ctx = fr->ctx;
    const int NT = fr->b.NT;
    if (obs_kf_bytes != 4 && obs_kf_bytes != 2) return fail(LCCRF_ERR_ARG, "obs_kf_bytes must be 4 (int32) or 2 (uint16)");
    if (obs_kf_bytes == 2 && nKF > 65536) return fail(LCCRF_ERR_ARG, "uint16 keyframe indices need nKF <= 65536");
    if (indexed) {
        if (!fr->kp_tab) return fail(LCCRF_ERR_STATE, "indexed observations need lccrf_frames_set_keyframe_keypoints first");
        if (nKF > fr->kp_cap) return fail(LCCRF_ERR_ARG, "nKF exceeds the keyframes of the resident keypoint table");
        if (obs_kf_bytes == 2 && fr->kp_stride > 65536) return fail(LCCRF_ERR_ARG, "uint16 feature indices need stride <= 65536");
    }
    if (NT > 0 && (!xyz || !obs_ptr || !kp2d)) return fail(LCCRF_ERR_ARG, "NULL argument");
    const long long nnz = NT > 0 ? obs_ptr[NT] : 0;
    if (NT > 0 && obs_ptr[0] != 0) return fail(LCCRF_ERR_ARG, "obs_ptr must start at 0");
    if (nnz > 0 && (!obs_kf || (!obs_uv && !indexed) || !kf_pose || !kf_intr || !kf_bounds || nKF <= 0))
        return fail(LCCRF_ERR_ARG, "NULL argument");
    // Tracking.cc:1858: points without observations never reach the CRF -- the caller drops them
    // (obs_ptr is host data, so this is a host-side structural check, not device work)
    for (int i = 0; i < NT; i++)
        if (obs_ptr[i + 1] <= obs_ptr[i]) return fail(LCCRF_ERR_ARG, "every point needs >= 1 observation (Tracking.cc:1858)");
    int slice_max = 0;
    if (kf_ptr) {
        if (kf_ptr[0] != 0 || kf_ptr[fr->b.B] != nKF) return fail(LCCRF_ERR_ARG, "kf_ptr must span [0, nKF]");
        for (int i = 0; i < fr->b.B; i++) {
            if (kf_ptr[i + 1] < kf_ptr[i]) return fail(LCCRF_ERR_ARG, "kf_ptr must be non-decreasing");
            if (kf_ptr[i + 1] - kf_ptr[i] > slice_max) slice_max = kf_ptr[i + 1] - kf_ptr[i];
        }
    }
    bool regraph = false;
    if (slice_max != in.kf_slice_max) regraph = true;  // the launch geometry of the unary kernel depends on it
    in.kf_slice_max = slice_max;
    {   // kernel parameters of the captured graph: a change of camera model needs a new capture
        float cam8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        const bool ucam = nnz > 0 && uniform_camera(kf_intr, kf_bounds, nKF, cam8);
        if (ucam != in.ucam || memcmp(cam8, in.cam8, sizeof(cam8)) != 0) regraph = true;
        in.ucam = ucam;
        memcpy(in.cam8, cam8, sizeof(cam8));
    }
    if (nnz > in.nnz_cap || !in.obs_kf || in.obs_kf_bytes != obs_kf_bytes || in.indexed != indexed) {
        dev_free(ctx, in.obs_kf);
        dev_free(ctx, in.obs_uv);
        in.obs_kf = nullptr;
        in.obs_uv = nullptr;
        const long long cap = nnz > in.nnz_cap ? nnz : in.nnz_cap;
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.obs_kf, (size_t)(cap ? cap : 1) * 8));  // up to an int32 {kf, fid} pair
        if (!indexed) LCCRF_TRY(dev_alloc(ctx, (void **)&in.obs_uv, (size_t)(cap ? cap : 1) * 8));
        in.nnz_cap = cap;
        regraph = true;
    }
    if (indexed && in.kp_gen != fr->kp_gen) regraph = true;  // the captured graph holds the table's address and stride
    in.kp_gen = fr->kp_gen;
    in.indexed = indexed;
    if (nKF > in.nKF_cap || !in.kf_pose) {
        dev_free(ctx, in.kf_pose);
        dev_free(ctx, in.kf_intr);
        dev_free(ctx, in.kf_bounds);
        dev_free(ctx, in.kf_packed);
        const size_t k = (size_t)(nKF ? nKF : 1);
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kf_pose, k * 48));
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kf_intr, k * 16));
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kf_bounds, k * 16));
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kf_packed, k * 80));
        in.nKF_cap = nKF;
        regraph = true;
    }
    if (!in.xyz) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.xyz, (size_t)(NT ? NT : 1) * 12));
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.obs_ptr, (size_t)(NT + 1) * 4));
        regraph = true;
    }
    if (!in.kp2d) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kp2d, (size_t)(NT ? NT : 1) * 8));
        regraph = true;
    }
    if (kf_ptr && !in.kf_ptr) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kf_ptr, (size_t)(fr->b.B + 1) * 4));
        regraph = true;
    }
    if (in.nKF != nKF || in.nnz != nnz || !in.from_map || in.visible || in.have_kf_ptr != (kf_ptr != nullptr)) regraph = true;
    in.visible = false;
    if (regraph) {
        graph_drop(in.graph);
        LCCRF_TRY(order_copies_after_alloc(ctx, in, st));  // every (re)allocation above sets regraph
    }
    in.nKF = nKF;
    in.nnz = nnz;
    in.obs_kf_bytes = obs_kf_bytes;
    in.have_kf_ptr = kf_ptr != nullptr;
    LCCRF_TRY(frames_upload_prior(fr, in, st));
    if (kf_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.kf_ptr, kf_ptr, (size_t)(fr->b.B + 1) * 4, cudaMemcpyHostToDevice, st));
    if (NT > 0) {
        LCCRF_CUDA(cudaMemcpyAsync(in.xyz, xyz, (size_t)NT * 12, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.obs_ptr, obs_ptr, (size_t)(NT + 1) * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kp2d, kp2d, (size_t)NT * 8, cudaMemcpyHostToDevice, st));
    }
    if (nnz > 0) {
        LCCRF_CUDA(cudaMemcpyAsync(in.obs_kf, obs_kf, (size_t)nnz * obs_kf_bytes * (indexed ? 2 : 1), cudaMemcpyHostToDevice, st));
        if (!indexed) LCCRF_CUDA(cudaMemcpyAsync(in.obs_uv, obs_uv, (size_t)nnz * 8, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kf_pose, kf_pose, (size_t)nKF * 48, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kf_intr, kf_intr, (size_t)nKF * 16, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kf_bounds, kf_bounds, (size_t)nKF * 16, cudaMemcpyHostToDevice, st));
    }
    in.from_map = true;
    in.have_inputs = true;
    return LCCRF_OK;
}

int lccrf_frames_set_inputs(lccrf_frames *fr, const float *observs, const float *error, const float *depth,
                            const float *kp2d) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    return frames_upload_direct(fr, fr->in[0], fr->ctx->stream, observs, error, depth, kp2d);
}

int lccrf_frames_set_map_inputs(lccrf_frames *fr, const float *xyz, const int *obs_ptr, const int *obs_kf,
                                const float *obs_uv, int nKF, const float *kf_pose, const float *kf_intr,
                                const float *kf_bounds, const float *kp2d, const int *kf_ptr) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    return frames_upload_map(fr, fr->in[0], fr->ctx->stream, xyz, obs_ptr, obs_kf, 4, obs_uv, nKF, kf_pose, kf_intr,
                             kf_bounds, kp2d, kf_ptr);
}

static int frames_enqueue(lccrf_frames *fr, FrameInputs &in) {
    Ctx *ctx = fr->ctx;
    Batch &b = fr->b;
    const int NT = b.NT;
    const lccrf_slam_params &prm = fr->prm;
    // the two pairwise kernels are independent until the first mean-field step: the smoothness kernel (keypoints
    // only) forks off before the unary, the appearance kernel follows the unary on the main branch
    LCCRF_TRY(ctx_fork(ctx));
    {
        // smoothKernel(N, w2, vpoints, vcorrd2d, mPoint3dStdev, mPoint2dStdev): 2-D branch   (Tracking.cc:1926)
        AuxScope aux(ctx);
        LCCRF_TRY(feat_div2(ctx, fr->feat2, in.kp2d, 2, prm.point2d_stdev, in.kp2d + 1, 2, prm.point2d_stdev, NT));
        LCCRF_TRY(lattice_set_build(ctx, b, b.lat[1], fr->feat2));
        LCCRF_TRY(potts_norm(ctx, b, b.lat[1]));
    }
    const float *observs = in.observs, *error = in.error, *depth = in.depth;
    if (in.visible) {
        DevMap *m = in.map;
        LCCRF_TRY(unary_map_points_visible(ctx, NT, in.vis, m->d_hdr, in.kf_bucket, fr->observs, fr->error, fr->depth, b.prob_ptr,
                                           in.have_kf_ptr ? in.kf_ptr : nullptr, b.B, in.kf_slice_max,
                                           in.ucam ? in.cam8 : nullptr));
        LCCRF_TRY(map_end_main_access(m));  // the map may change from here on (the next step's delta, on the map's stream)
        observs = fr->observs;
        error = fr->error;
        depth = fr->depth;
    } else if (in.from_map) {
        LCCRF_TRY(unary_pack_kf(ctx, in.kf_packed, in.kf_pose, in.kf_intr, in.kf_bounds, in.nKF));
        LCCRF_TRY(unary_map_points_packed(ctx, NT, in.nKF, in.xyz, in.obs_ptr, in.obs_kf, in.obs_kf_bytes, in.obs_uv,
                                          in.kf_packed, fr->observs, fr->error, fr->depth, b.prob_ptr,
                                          in.have_kf_ptr ? in.kf_ptr : nullptr, b.B, in.kf_slice_max,
                                          in.ucam ? in.cam8 : nullptr, in.indexed ? fr->kp_tab : nullptr, fr->kp_stride));
        observs = fr->observs;
        error = fr->error;
        depth = fr->depth;
    }
    // RroughClassify -> setUnaryEnergyFromLabel   (Tracking.cc:1871,1921)
    LCCRF_TRY(unary_classify(ctx, NT, observs, error, depth, in.use_p4 ? in.p4 : nullptr, prm, fr->label,
                             in.use_p4_has ? in.p4_has : nullptr, b.prob_ptr, b.B));
    LCCRF_TRY(mf_unary_from_label(ctx, b.unary, fr->label, NT, 2, fr->energies[0], fr->d_en, fr->d_en + 2));
    // appearanceKernel(N, w1, vobservs, verrors, mObservStdev, mRpjErrorStdev)   (Tracking.cc:1923)
    LCCRF_TRY(feat_div2(ctx, fr->feat, observs, 1, prm.stdev_beta, error, 1, prm.stdev_alpha, NT));
    LCCRF_TRY(lattice_set_build(ctx, b, b.lat[0], fr->feat));
    LCCRF_TRY(potts_norm(ctx, b, b.lat[0]));
    LCCRF_TRY(ctx_join(ctx));
    // inference(iters, true)   (Tracking.cc:1929)
    LCCRF_TRY(mf_start(ctx, b));
    for (int it = 0; it < prm.iters; it++) LCCRF_TRY(mf_step(ctx, b, 1.0f));
    LCCRF_TRY(mf_build_map(ctx, b));
    return LCCRF_OK;
}

// run the batch from input set `in` on ctx->stream: CUDA-graph replay when enabled
static int frames_run_slot(lccrf_frames *fr, FrameInputs &in) {
    Ctx *ctx = fr->ctx;
    if (!in.have_inputs) return fail(LCCRF_ERR_STATE, "frames_run before set_inputs");
    if (in.has_delta) {
        // this step's map changes: plain launches on the map's own stream, behind the upload and behind the previous
        // step's unary -- they run beside that step's lattice builds and mean-field iterations
        in.has_delta = false;
        LCCRF_CUDA(cudaStreamWaitEvent(in.map->mstream, in.up_done, 0));
        {
            MapStreamScope on_map_stream(in.map);
            LCCRF_TRY(map_apply_dev(in.map, in.delta, nullptr));
        }
        LCCRF_TRY(map_end_async_mut(in.map));
    }
    if (in.visible) LCCRF_TRY(map_begin_main_access(in.map));
    if (ctx->opt_graphs && !ctx->opt_profile && in.indexed && in.kp_gen != fr->kp_gen) {
        // the keypoint table moved (keyframes inserted) since this slot was captured
        graph_drop(in.graph);
        in.kp_gen = fr->kp_gen;
    }
    LCCRF_TRY(graph_run(ctx, in.graph, [&] { return frames_enqueue(fr, in); }));
    fr->ran = true;
    return LCCRF_OK;
}

int lccrf_frames_run(lccrf_frames *fr) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    fr->last_slot = 0;
    return frames_run_slot(fr, fr->in[0]);
}

int lccrf_frames_get_outputs(lccrf_frames *fr, short *map, float *prob) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (!fr->ran) return fail(LCCRF_ERR_STATE, "frames_get_outputs before frames_run");
    for (int s_ = 0; s_ < 2; s_++)
        if (fr->in[s_].in_flight)
            return fail(LCCRF_ERR_STATE, "a pipelined submission is in flight: its results go to the buffers given to "
                                         "lccrf_frames_submit_* / lccrf_frames_set_partition_outputs; wait for both slots first");
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)fr->b.NT;
    if (n && map) LCCRF_CUDA(cudaMemcpyAsync(map, fr->b.map, n * 2, cudaMemcpyDeviceToHost, ctx->stream));
    if (n && prob) LCCRF_CUDA(cudaMemcpyAsync(prob, fr->b.cur, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return check_status(ctx);
}

// ---- pipelined end-to-end submission (two input slots) ----
static int frames_submit_prologue(lccrf_frames *fr, int slot, FrameInputs **in_out) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (slot < 0 || slot > 1) return fail(LCCRF_ERR_ARG, "slot must be 0 or 1");
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->copy_stream) LCCRF_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    FrameInputs &in = fr->in[slot];
    if (in.in_flight) return fail(LCCRF_ERR_STATE, "slot still in flight: call lccrf_frames_wait first");
    if (!in.up_done) {
        LCCRF_CUDA(cudaEventCreateWithFlags(&in.up_done, cudaEventDisableTiming));
        LCCRF_CUDA(cudaEventCreateWithFlags(&in.run_done, cudaEventDisableTiming));
        LCCRF_CUDA(cudaEventCreateWithFlags(&in.out_done, cudaEventDisableTiming));
        LCCRF_CUDA(cudaEventRecord(in.run_done, ctx->stream));
        LCCRF_CUDA(cudaHostAlloc((void **)&in.h_status, sizeof(int), cudaHostAllocDefault));
        *in.h_status = 0;
    }
    // the copy stream may overwrite this slot only after the last run that read it
    LCCRF_CUDA(cudaStreamWaitEvent(ctx->copy_stream, in.run_done, 0));
    *in_out = &in;
    return LCCRF_OK;
}

static int frames_submit_epilogue(lccrf_frames *fr, int slot, FrameInputs &in, short *map_out, float *prob_out) {
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaEventRecord(in.up_done, ctx->copy_stream));
    LCCRF_CUDA(cudaStreamWaitEvent(ctx->stream, in.up_done, 0));
    if (graph_will_capture(ctx, in.graph)) {
        // the capture pass synchronises; make sure the upload has landed first
        LCCRF_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    }
    LCCRF_TRY(frames_run_slot(fr, in));
    LCCRF_CUDA(cudaEventRecord(in.run_done, ctx->stream));
    // Results leave through per-slot device staging on a third stream: the next slot's run neither waits for the PCIe
    // copy nor overwrites labels / marginals that are still on their way out.
    const size_t n = (size_t)fr->b.NT;
    if (!ctx->d2h_stream) LCCRF_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
    if (!in.out_stage) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.out_stage, (n ? n : 1) * 10 + 256));
        LCCRF_CUDA(cudaEventCreateWithFlags(&in.res_ready, cudaEventDisableTiming));
    }
    char *st_prob = (char *)in.out_stage, *st_map = st_prob + n * 8, *st_status = st_map + ((n * 2 + 15) / 16) * 16;
    if (n && map_out) LCCRF_CUDA(cudaMemcpyAsync(st_map, fr->b.map, n * 2, cudaMemcpyDeviceToDevice, ctx->stream));
    if (n && prob_out) LCCRF_CUDA(cudaMemcpyAsync(st_prob, fr->b.cur, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    LCCRF_CUDA(cudaMemcpyAsync(st_status, ctx->d_status, sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream));
    if (in.part_dyn_ptr || in.part_dyn || in.part_stat_ptr || in.part_stat) {
        // label application of THIS submission (Tracking.cc:1945-1955), before the other slot's run reuses the labels
        const int NT = fr->b.NT, B = fr->b.B;
        const size_t nB = (size_t)(B + 1), nT = (size_t)(NT > 0 ? NT : 1);
        if (!fr->part)
            LCCRF_TRY(dev_alloc(ctx, (void **)&fr->part, (2 * nB + 3 * nT) * sizeof(int) + label_partition_scratch_bytes(NT)));
        int *d_dyn_ptr = fr->part, *d_stat_ptr = d_dyn_ptr + nB, *d_dyn = d_stat_ptr + nB, *d_stat = d_dyn + nT,
            *d_fid = d_stat + nT, *d_scratch = d_fid + nT;
        cudaStream_t st = ctx->stream;
        if (in.part_fid && NT) LCCRF_CUDA(cudaMemcpyAsync(d_fid, in.part_fid, (size_t)NT * 4, cudaMemcpyHostToDevice, st));
        LCCRF_TRY(label_partition(ctx, fr->b.map, NT, fr->b.prob_ptr, B, in.part_fid ? d_fid : nullptr, d_scratch, d_dyn_ptr,
                                  d_dyn, d_stat_ptr, d_stat));
        if (in.part_dyn_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.part_dyn_ptr, d_dyn_ptr, nB * 4, cudaMemcpyDeviceToHost, st));
        if (in.part_stat_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.part_stat_ptr, d_stat_ptr, nB * 4, cudaMemcpyDeviceToHost, st));
        if (in.part_dyn && NT) LCCRF_CUDA(cudaMemcpyAsync(in.part_dyn, d_dyn, (size_t)NT * 4, cudaMemcpyDeviceToHost, st));
        if (in.part_stat && NT) LCCRF_CUDA(cudaMemcpyAsync(in.part_stat, d_stat, (size_t)NT * 4, cudaMemcpyDeviceToHost, st));
    }
    LCCRF_CUDA(cudaEventRecord(in.res_ready, ctx->stream));
    LCCRF_CUDA(cudaStreamWaitEvent(ctx->d2h_stream, in.res_ready, 0));
    if (n && map_out) LCCRF_CUDA(cudaMemcpyAsync(map_out, st_map, n * 2, cudaMemcpyDeviceToHost, ctx->d2h_stream));
    if (n && prob_out) LCCRF_CUDA(cudaMemcpyAsync(prob_out, st_prob, n * 8, cudaMemcpyDeviceToHost, ctx->d2h_stream));
    LCCRF_CUDA(cudaMemcpyAsync(in.h_status, st_status, sizeof(int), cudaMemcpyDeviceToHost, ctx->d2h_stream));
    LCCRF_CUDA(cudaEventRecord(in.out_done, ctx->d2h_stream));
    in.in_flight = true;
    fr->last_slot = slot;
    return LCCRF_OK;
}

int lccrf_frames_submit_map(lccrf_frames *fr, int slot, const float *xyz, const int *obs_ptr, const void *obs_kf,
                            int obs_kf_bytes, const float *obs_uv, int nKF, const float *kf_pose, const float *kf_intr,
                            const float *kf_bounds, const float *kp2d, const int *kf_ptr, short *map_out,
                            float *prob_out) {
    FrameInputs *in = nullptr;
    LCCRF_TRY(frames_submit_prologue(fr, slot, &in));
    LCCRF_TRY(frames_upload_map(fr, *in, fr->ctx->copy_stream, xyz, obs_ptr, obs_kf, obs_kf_bytes, obs_uv, nKF, kf_pose,
                                kf_intr, kf_bounds, kp2d, kf_ptr));
    return frames_submit_epilogue(fr, slot, *in, map_out, prob_out);
}

// ---- resident keyframe keypoints + indexed observations ----
int lccrf_frames_set_keyframe_keypoints(lccrf_frames *fr, int kf_first, int kf_count, int stride, const float *kp_uv) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (kf_first < 0 || kf_count < 0 || stride <= 0) return fail(LCCRF_ERR_ARG, "bad keyframe range or stride");
    if (kf_count > 0 && !kp_uv) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (fr->kp_tab && stride != fr->kp_stride) return fail(LCCRF_ERR_ARG, "stride differs from the resident table's");
    for (int s = 0; s < 2; s++)
        if (fr->in[s].in_flight) return fail(LCCRF_ERR_STATE, "a submission is in flight: call lccrf_frames_wait first");
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const long long need = (long long)kf_first + kf_count;
    if (need > 0x7fffffffLL) return fail(LCCRF_ERR_ARG, "too many keyframes");
    if (!fr->kp_tab || need > fr->kp_cap) {
        long long cap = fr->kp_cap ? 2LL * fr->kp_cap : 0;
        if (cap < need) cap = need;
        if (cap < 1) cap = 1;
        float *nt = nullptr;
        LCCRF_TRY(dev_alloc(ctx, (void **)&nt, (size_t)cap * stride * 8, true));
        if (fr->kp_tab)
            LCCRF_CUDA(cudaMemcpyAsync(nt, fr->kp_tab, (size_t)fr->kp_cap * stride * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        dev_free(ctx, fr->kp_tab);
        fr->kp_tab = nt;
        fr->kp_cap = (int)cap;
        fr->kp_stride = stride;
        fr->kp_gen++;
    }
    if (kf_count > 0)
        LCCRF_CUDA(cudaMemcpyAsync(fr->kp_tab + (size_t)kf_first * stride * 2, kp_uv, (size_t)kf_count * stride * 8,
                                   cudaMemcpyHostToDevice, ctx->stream));
    // rare call (keyframe insertion): synchronise so that the host buffer is free on return and the copy stream of
    // the pipelined submissions sees the table
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

int lccrf_frames_set_map_inputs_indexed(lccrf_frames *fr, const float *xyz, const int *obs_ptr, const void *obs_ref,
                                        int index_bytes, int nKF, const float *kf_pose, const float *kf_intr,
                                        const float *kf_bounds, const float *kp2d, const int *kf_ptr) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    return frames_upload_map(fr, fr->in[0], fr->ctx->stream, xyz, obs_ptr, obs_ref, index_bytes, nullptr, nKF, kf_pose,
                             kf_intr, kf_bounds, kp2d, kf_ptr, true);
}

int lccrf_frames_submit_map_indexed(lccrf_frames *fr, int slot, const float *xyz, const int *obs_ptr, const void *obs_ref,
                                    int index_bytes, int nKF, const float *kf_pose, const float *kf_intr,
                                    const float *kf_bounds, const float *kp2d, const int *kf_ptr, short *map_out,
                                    float *prob_out) {
    FrameInputs *in = nullptr;
    LCCRF_TRY(frames_submit_prologue(fr, slot, &in));
    LCCRF_TRY(frames_upload_map(fr, *in, fr->ctx->copy_stream, xyz, obs_ptr, obs_ref, index_bytes, nullptr, nKF, kf_pose,
                                kf_intr, kf_bounds, kp2d, kf_ptr, true));
    return frames_submit_epilogue(fr, slot, *in, map_out, prob_out);
}

int lccrf_frames_submit(lccrf_frames *fr, int slot, const float *observs, const float *error, const float *depth,
                        const float *kp2d, short *map_out, float *prob_out) {
    FrameInputs *in = nullptr;
    LCCRF_TRY(frames_submit_prologue(fr, slot, &in));
    LCCRF_TRY(frames_upload_direct(fr, *in, fr->ctx->copy_stream, observs, error, depth, kp2d));
    return frames_submit_epilogue(fr, slot, *in, map_out, prob_out);
}

int lccrf_frames_wait(lccrf_frames *fr, int slot) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (slot < 0 || slot > 1) return fail(LCCRF_ERR_ARG, "slot must be 0 or 1");
    FrameInputs &in = fr->in[slot];
    if (!in.in_flight) return LCCRF_OK;
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    LCCRF_CUDA(cudaEventSynchronize(in.out_done));
    in.in_flight = false;
    if (*in.h_status) {
        cudaMemsetAsync(fr->ctx->d_status, 0, sizeof(int), fr->ctx->stream);
        return decode_status(*in.h_status);
    }
    return LCCRF_OK;
}

int lccrf_frames_get_debug(lccrf_frames *fr, short *init_label, float *observs, float *error, float *depth, int *V) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (!fr->ran) return fail(LCCRF_ERR_STATE, "frames_get_debug before frames_run");
    for (int s_ = 0; s_ < 2; s_++)
        if (fr->in[s_].in_flight)
            return fail(LCCRF_ERR_STATE, "a pipelined submission is in flight: its results go to the buffers given to "
                                         "lccrf_frames_submit_* / lccrf_frames_set_partition_outputs; wait for both slots first");
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)fr->b.NT;
    cudaStream_t st = ctx->stream;
    const FrameInputs &in = fr->in[fr->last_slot];
    const float *d_obs = in.from_map ? fr->observs : in.observs, *d_err = in.from_map ? fr->error : in.error,
                *d_dep = in.from_map ? fr->depth : in.depth;
    if (n && init_label) LCCRF_CUDA(cudaMemcpyAsync(init_label, fr->label, n * 2, cudaMemcpyDeviceToHost, st));
    if (n && observs) LCCRF_CUDA(cudaMemcpyAsync(observs, d_obs, n * 4, cudaMemcpyDeviceToHost, st));
    if (n && error) LCCRF_CUDA(cudaMemcpyAsync(error, d_err, n * 4, cudaMemcpyDeviceToHost, st));
    if (n && depth) LCCRF_CUDA(cudaMemcpyAsync(depth, d_dep, n * 4, cudaMemcpyDeviceToHost, st));
    std::vector<int> vb[2];
    if (V) {
        for (int k = 0; k < 2; k++) {
            vb[k].resize(fr->b.B + 1);
            LCCRF_CUDA(cudaMemcpyAsync(vb[k].data(), fr->b.lat[k]->vbase, (size_t)(fr->b.B + 1) * 4, cudaMemcpyDeviceToHost, st));
        }
    }
    LCCRF_CUDA(cudaStreamSynchronize(st));
    if (V)
        for (int i = 0; i < fr->b.B; i++)
            for (int k = 0; k < 2; k++) V[2 * i + k] = vb[k][i + 1] - vb[k][i];
    return LCCRF_OK;
}

// label application (Tracking.cc:1945-1955): stable partition of the batch's MAP labels
int lccrf_frames_partition(lccrf_frames *fr, const int *fid, int *dyn_ptr, int *dyn_list, int *stat_ptr, int *stat_list) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (!fr->ran) return fail(LCCRF_ERR_STATE, "frames_partition before frames_run");
    for (int s_ = 0; s_ < 2; s_++)
        if (fr->in[s_].in_flight)
            return fail(LCCRF_ERR_STATE, "a pipelined submission is in flight: its results go to the buffers given to "
                                         "lccrf_frames_submit_* / lccrf_frames_set_partition_outputs; wait for both slots first");
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const int NT = fr->b.NT, B = fr->b.B;
    const size_t nB = (size_t)(B + 1), nT = (size_t)(NT > 0 ? NT : 1);
    if (!fr->part)
        LCCRF_TRY(dev_alloc(ctx, (void **)&fr->part, (2 * nB + 3 * nT) * sizeof(int) + label_partition_scratch_bytes(NT)));
    int *d_dyn_ptr = fr->part, *d_stat_ptr = d_dyn_ptr + nB, *d_dyn = d_stat_ptr + nB, *d_stat = d_dyn + nT,
        *d_fid = d_stat + nT, *d_scratch = d_fid + nT;
    cudaStream_t st = ctx->stream;
    if (fid && NT) LCCRF_CUDA(cudaMemcpyAsync(d_fid, fid, (size_t)NT * 4, cudaMemcpyHostToDevice, st));
    LCCRF_TRY(label_partition(ctx, fr->b.map, NT, fr->b.prob_ptr, B, fid ? d_fid : nullptr, d_scratch, d_dyn_ptr, d_dyn,
                              d_stat_ptr, d_stat));
    std::vector<int> hp(2 * nB);
    LCCRF_CUDA(cudaMemcpyAsync(hp.data(), d_dyn_ptr, 2 * nB * sizeof(int), cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));
    const int n_dyn = hp[B], n_stat = hp[nB + B];
    if (n_dyn < 0 || n_stat < 0 || n_dyn + n_stat != NT) return fail(LCCRF_ERR_STATE, "label partition is inconsistent");
    if (dyn_ptr) memcpy(dyn_ptr, hp.data(), nB * sizeof(int));
    if (stat_ptr) memcpy(stat_ptr, hp.data() + nB, nB * sizeof(int));
    if (dyn_list && n_dyn) LCCRF_CUDA(cudaMemcpyAsync(dyn_list, d_dyn, (size_t)n_dyn * 4, cudaMemcpyDeviceToHost, st));
    if (stat_list && n_stat) LCCRF_CUDA(cudaMemcpyAsync(stat_list, d_stat, (size_t)n_stat * 4, cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));
    return LCCRF_OK;
}

int lccrf_frames_debug_counters(lccrf_frames *fr, int k, int *out8) {
    if (!fr || !out8) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (k < 0 || k >= (int)fr->b.lat.size()) return fail(LCCRF_ERR_ARG, "lattice index out of range");
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    LCCRF_CUDA(cudaMemcpyAsync(out8, fr->b.lat[k]->row_counts, 8 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

// SURVEY.md 8(d) formulas with the actual V of every problem
int lccrf_frames_algorithmic_bytes(lccrf_frames *fr, double *total, double *per_iteration, double *unary) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    std::vector<int> V((size_t)fr->b.B * 2);
    LCCRF_TRY(lccrf_frames_get_debug(fr, nullptr, nullptr, nullptr, nullptr, V.data()));
    const double d = 2, D = 3, L = 2, K = 2, T = fr->prm.iters;
    double tot = 0, it_tot = 0;
    for (int i = 0; i < fr->b.B; i++) {
        const double N = fr->b.h_prob_ptr[i + 1] - fr->b.h_prob_ptr[i];
        double Bit = K * N * 4 + 2 * N * L * 4, Bb = 0;
        for (int k = 0; k < 2; k++) {
            const double Vk = V[2 * i + k];
            auto Bf = [&](double l) { return 2 * N * D * 8 + 2 * N * l * 4 + D * Vk * (2 * l * 4 + 8); };
            Bit += Bf(L);
            Bb += N * d * 4 + N * D * 8 + Vk * (2 * d + 8 * D) + Bf(1) + N * 4;
        }
        tot += N * 2 + N * L * 4 + 2 * N * L * 4 + Bb + T * Bit + N * L * 4 + N * 2;
        it_tot += Bit;
    }
    double u = 0;
    const FrameInputs &in = fr->in[fr->last_slot];
    long long nnz = in.nnz;
    if (in.visible && fr->b.NT > 0) {  // observations of the visible points: counted on the device
        Ctx *ctx = fr->ctx;
        int *d_cnt = nullptr;
        LCCRF_TRY(dev_alloc(ctx, (void **)&d_cnt, (size_t)fr->b.NT * 4));
        int rc = map_export_dev(in.map, fr->b.NT, in.vis, d_cnt);
        std::vector<int> cnt((size_t)fr->b.NT);
        if (rc == LCCRF_OK) {
            cudaError_t e = cudaMemcpyAsync(cnt.data(), d_cnt, cnt.size() * 4, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
        }
        dev_free(ctx, d_cnt);
        LCCRF_TRY(rc);
        nnz = 0;
        for (int c : cnt) nnz += c;
    }
    if (in.from_map) u = (double)nnz * 12 + (double)fr->b.NT * 24 + (double)in.nKF * 80;
    if (total) *total = tot + u;
    if (per_iteration) *per_iteration = it_tot;
    if (unary) *unary = u;
    return LCCRF_OK;
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

// bytes of the staged arrays of a delta (every array 256-byte aligned); with_keypoints = false when the new keyframes'
// keypoints are copied straight from the host array
static size_t delta_stage_bytes(const lccrf_map_delta &d, int kp_stride, bool with_keypoints) {
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    size_t n = 0;
    n += al((size_t)d.kf_count * 48) + al((size_t)d.kf_count * 16) * 2;
    if (with_keypoints && d.kf_keypoints) n += al((size_t)d.kf_count * kp_stride * 8);
    n += al((size_t)d.n_pose * 4) + al((size_t)d.n_pose * 48);
    n += al((size_t)d.n_xyz * 4) + al((size_t)d.n_xyz * 12);
    n += al((size_t)d.n_erase * 4) * 2 + al((size_t)d.n_bad * 4) + al((size_t)d.n_add * 4) * 3;
    return n + 256;
}

// copy the delta's host arrays to `base` on stream st and describe them in `out`
static int delta_stage(const lccrf_map_delta &d, int kp_stride, bool with_keypoints, char *base, cudaStream_t st, DeltaDev *out) {
    size_t off = 0;
    cudaError_t err = cudaSuccess;
    auto put = [&](const void *src, size_t bytes) -> const void * {
        if (!src || bytes == 0) return nullptr;
        char *dst = base + off;
        off += (bytes + 255) / 256 * 256;
        cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) err = e;
        return dst;
    };
    DeltaDev o;
    o.kf_first = d.kf_first;
    o.kf_count = d.kf_count;
    o.kf_pose = (const float *)put(d.kf_pose, (size_t)d.kf_count * 48);
    o.kf_intr = (const float *)put(d.kf_intr, (size_t)d.kf_count * 16);
    o.kf_bounds = (const float *)put(d.kf_bounds, (size_t)d.kf_count * 16);
    if (with_keypoints) o.kf_keypoints = (const float *)put(d.kf_keypoints, (size_t)d.kf_count * kp_stride * 8);
    o.n_pose = d.n_pose;
    o.pose_kf = (const int *)put(d.pose_kf, (size_t)d.n_pose * 4);
    o.pose = (const float *)put(d.pose, (size_t)d.n_pose * 48);
    o.n_xyz = d.n_xyz;
    o.xyz_id = (const int *)put(d.xyz_id, (size_t)d.n_xyz * 4);
    o.xyz = (const float *)put(d.xyz, (size_t)d.n_xyz * 12);
    o.n_erase = d.n_erase;
    o.erase_pt = (const int *)put(d.erase_pt, (size_t)d.n_erase * 4);
    o.erase_kf = (const int *)put(d.erase_kf, (size_t)d.n_erase * 4);
    o.n_bad = d.n_bad;
    o.bad_pt = (const int *)put(d.bad_pt, (size_t)d.n_bad * 4);
    o.n_add = d.n_add;
    o.add_pt = (const int *)put(d.add_pt, (size_t)d.n_add * 4);
    o.add_kf = (const int *)put(d.add_kf, (size_t)d.n_add * 4);
    o.add_fid = (const int *)put(d.add_fid, (size_t)d.n_add * 4);
    if (d.n_erase_seg > 0) o.erase_seg.assign(d.erase_seg_ptr, d.erase_seg_ptr + d.n_erase_seg + 1);
    if (d.n_add_seg > 0) o.add_seg.assign(d.add_seg_ptr, d.add_seg_ptr + d.n_add_seg + 1);
    if (err != cudaSuccess) return fail(LCCRF_ERR_CUDA, std::string("map delta upload: ") + cudaGetErrorString(err));
    *out = o;
    return LCCRF_OK;
}

// explicit point ids name points the caller creates densely: raise the capacity to the largest id of the delta
static int delta_grow_points(DevMap *m, const lccrf_map_delta &d) {
    if (d.n_xyz > 0 && d.xyz_id) {
        int mx = -1;
        for (int i = 0; i < d.n_xyz; i++) {
            if (d.xyz_id[i] < 0) return fail(LCCRF_ERR_ARG, "map delta: negative point id");
            if (d.xyz_id[i] > mx) mx = d.xyz_id[i];
        }
        LCCRF_TRY(map_reserve_points(m, mx + 1));
        if (mx + 1 > m->n_pt) m->n_pt = mx + 1;
    }
    return LCCRF_OK;
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

// ---- frame batches against the resident map ----
static int frames_upload_visible(lccrf_frames *fr, FrameInputs &in, cudaStream_t st, lccrf_map *map, const lccrf_map_delta *delta,
                                 const int *point_id, const float *kp2d, const int *kf_ptr) {
    Ctx *ctx = fr->ctx;
    if (!map || !map->m) return fail(LCCRF_ERR_ARG, "map is NULL");
    DevMap *m = map->m;
    if (m->ctx != ctx) return fail(LCCRF_ERR_ARG, "map and frames belong to different contexts");
    const int NT = fr->b.NT, B = fr->b.B;
    if (NT > 0 && (!point_id || !kp2d)) return fail(LCCRF_ERR_ARG, "NULL argument");
    const bool pipelined = st != ctx->stream;
    bool regraph = false, fresh = false;
    if (delta && pipelined) {
        // host-side bookkeeping + capacity growth, stream-ordered on the MAP's stream behind the last access of the
        // context's stream (an array that moves is freed there, and the previous step's unary may still read it)
        LCCRF_TRY(map_begin_async_mut(m));
        MapStreamScope on_map_stream(m);
        LCCRF_TRY(map_prepare(m, *delta));
        LCCRF_TRY(delta_grow_points(m, *delta));
    } else if (delta) {
        LCCRF_TRY(map_begin_main_access(m));
        LCCRF_TRY(map_prepare(m, *delta));
        LCCRF_TRY(delta_grow_points(m, *delta));
    }
    if (delta) {
        const size_t need = delta_stage_bytes(*delta, m->kp_stride, true);
        if (need > in.stage_cap) {
            // rare (first steps): cudaFree waits for the device, so nothing still reads the old block
            if (in.stage) LCCRF_CUDA(cudaFree(in.stage));
            in.stage = nullptr;
            in.stage_cap = 0;
            const size_t cap = need + need / 2;
            LCCRF_CUDA(cudaMalloc(&in.stage, cap));
            in.stage_cap = cap;
        }
    }
    if (m->n_kf <= 0 && NT > 0) return fail(LCCRF_ERR_STATE, "the map has no keyframes");
    int slice_max = 0;
    if (kf_ptr) {
        if (kf_ptr[0] != 0 || kf_ptr[B] != m->n_kf) return fail(LCCRF_ERR_ARG, "kf_ptr must span [0, number of keyframes]");
        for (int i = 0; i < B; i++) {
            if (kf_ptr[i + 1] < kf_ptr[i]) return fail(LCCRF_ERR_ARG, "kf_ptr must be non-decreasing");
            if (kf_ptr[i + 1] - kf_ptr[i] > slice_max) slice_max = kf_ptr[i + 1] - kf_ptr[i];
        }
    }
    if (slice_max != in.kf_slice_max) regraph = true;
    in.kf_slice_max = slice_max;
    {   // camera model and shared-memory keyframe slots are kernel parameters of the captured graph
        const bool ucam = m->cam_set && m->ucam;
        if (ucam != in.ucam || (ucam && memcmp(m->cam8, in.cam8, sizeof(in.cam8)) != 0)) regraph = true;
        in.ucam = ucam;
        memcpy(in.cam8, m->cam8, sizeof(in.cam8));
        int bucket = (m->n_kf + 127) / 128 * 128;
        if (bucket != in.kf_bucket) regraph = true;
        in.kf_bucket = bucket;
    }
    if (!in.vis) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.vis, (size_t)(NT ? NT : 1) * 4));
        regraph = fresh = true;
    }
    if (!in.kp2d) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kp2d, (size_t)(NT ? NT : 1) * 8));
        regraph = fresh = true;
    }
    if (kf_ptr && !in.kf_ptr) {
        LCCRF_TRY(dev_alloc(ctx, (void **)&in.kf_ptr, (size_t)(B + 1) * 4));
        regraph = fresh = true;
    }
    if (!in.visible || in.map != m || in.have_kf_ptr != (kf_ptr != nullptr)) regraph = true;
    if (regraph) graph_drop(in.graph);
    if (fresh) LCCRF_TRY(order_copies_after_alloc(ctx, in, st));
    in.visible = true;
    in.from_map = true;
    in.indexed = false;
    in.map = m;
    in.have_kf_ptr = kf_ptr != nullptr;
    in.nKF = m->n_kf;
    in.nnz = -1;
    LCCRF_TRY(frames_upload_prior(fr, in, st));
    in.has_delta = false;
    if (delta) {
        if (pipelined) {
            LCCRF_TRY(delta_stage(*delta, m->kp_stride, true, (char *)in.stage, st, &in.delta));
            in.has_delta = true;  // applied on the context's stream once the upload has landed (frames_run_slot)
        } else {
            DeltaDev dd;
            LCCRF_TRY(delta_stage(*delta, m->kp_stride, false, (char *)in.stage, st, &dd));
            LCCRF_TRY(map_apply_dev(m, dd, delta->kf_count > 0 ? delta->kf_keypoints : nullptr));
        }
    }
    if (kf_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.kf_ptr, kf_ptr, (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, st));
    if (NT > 0) {
        LCCRF_CUDA(cudaMemcpyAsync(in.vis, point_id, (size_t)NT * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kp2d, kp2d, (size_t)NT * 8, cudaMemcpyHostToDevice, st));
    }
    in.have_inputs = true;
    return LCCRF_OK;
}

int lccrf_frames_set_visible(lccrf_frames *fr, lccrf_map *map, const lccrf_map_delta *delta, const int *point_id,
                             const float *kp2d, const int *kf_ptr) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    for (int s_ = 0; s_ < 2; s_++)
        if (fr->in[s_].in_flight) return fail(LCCRF_ERR_STATE, "a submission is in flight: call lccrf_frames_wait first");
    LCCRF_TRY(frames_upload_visible(fr, fr->in[0], fr->ctx->stream, map, delta, point_id, kp2d, kf_ptr));
    // the host arrays (delta included) are free on return
    LCCRF_CUDA(cudaStreamSynchronize(fr->ctx->stream));
    return LCCRF_OK;
}

int lccrf_frames_submit_visible(lccrf_frames *fr, int slot, lccrf_map *map, const lccrf_map_delta *delta, const int *point_id,
                                const float *kp2d, const int *kf_ptr, short *map_out, float *prob_out) {
    FrameInputs *in = nullptr;
    PhaseTimer tm(fr && fr->ctx->opt_trace);
    LCCRF_TRY(frames_submit_prologue(fr, slot, &in));
    tm.mark("prologue");
    LCCRF_TRY(frames_upload_visible(fr, *in, fr->ctx->copy_stream, map, delta, point_id, kp2d, kf_ptr));
    tm.mark("upload");
    const int rc = frames_submit_epilogue(fr, slot, *in, map_out, prob_out);
    tm.mark("apply+run+results");
    return rc;
}

int lccrf_frames_set_prior(lccrf_frames *fr, int slot, const double *p4, const unsigned char *has_prior) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (slot < 0 || slot > 1) return fail(LCCRF_ERR_ARG, "slot must be 0 or 1");
    if (!p4 && has_prior) return fail(LCCRF_ERR_ARG, "has_prior without p4");
    fr->in[slot].h_p4 = p4;
    fr->in[slot].h_p4_has = has_prior;
    return LCCRF_OK;
}

int lccrf_frames_set_partition_outputs(lccrf_frames *fr, int slot, const int *fid, int *dyn_ptr, int *dyn_list, int *stat_ptr,
                                       int *stat_list) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (slot < 0 || slot > 1) return fail(LCCRF_ERR_ARG, "slot must be 0 or 1");
    FrameInputs &in = fr->in[slot];
    if (in.in_flight) return fail(LCCRF_ERR_STATE, "slot still in flight: call lccrf_frames_wait first");
    in.part_fid = fid;
    in.part_dyn_ptr = dyn_ptr;
    in.part_dyn = dyn_list;
    in.part_stat_ptr = stat_ptr;
    in.part_stat = stat_list;
    return LCCRF_OK;
}

}  // extern "C"
