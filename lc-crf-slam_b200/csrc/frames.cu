// frames.cu -- lccrf_frames: B independent per-frame CRFs (Tracking.cc:1871-1930) in one launch sequence.  A step's
// inputs come as the per-frame vectors, as a map snapshot (flat or indexed observations) or as ids of a device-resident
// map's points; they go through the synchronous path (set_* + run) or the pipelined one (submit_* + wait, two slots).
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "engine.cuh"

using namespace lccrf;

namespace {

// where the unary inputs of a run come from
enum class FrameSource {
    kDirect,           // the Tracking.cc:1849-1870 vectors (lccrf_frames_set_inputs / submit)
    kSnapshot,         // a map snapshot with keyframe indices and keypoints (set_map_inputs / submit_map)
    kSnapshotIndexed,  // a map snapshot with {keyframe, feature index} pairs; keypoints from lccrf_frames::kp_tab
    kVisible,          // ids of a device-resident map's points (set_visible / submit_visible)
};

// Everything frames_enqueue passes to a kernel that can differ between runs of one frames object.  A captured graph
// holds these values: a slot replays its graph only while the next run's key equals the key it was captured for.
// Fields the source does not read keep their defaults.
struct FrameLaunch {
    FrameSource src = FrameSource::kDirect;
    // slot arrays the run reads
    const float *observs = nullptr, *error = nullptr, *depth = nullptr, *kp2d = nullptr;
    const float *xyz = nullptr, *obs_uv = nullptr, *kf_pose = nullptr, *kf_intr = nullptr, *kf_bounds = nullptr;
    const int *obs_ptr = nullptr, *vis = nullptr;
    const void *obs_kf = nullptr;
    void *kf_packed = nullptr;
    const int *kf_ptr = nullptr;  // [B+1] keyframe slice of each problem, or null
    int nKF = 0, obs_kf_bytes = 0;
    long long nnz = 0;     // no kernel takes it, but a change has always meant a new capture
    int kf_slice_max = 0;  // largest per-problem keyframe slice (0 = unknown)
    int kf_bucket = 0;     // shared-memory keyframe slots of the visible unary
    bool ucam = false;     // every keyframe has the same intrinsics / image bounds: cam8 (all zero otherwise)
    float cam8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    DevMap *map = nullptr;
    const float *kp_tab = nullptr;  // resident keypoint table (indexed source), read when the run starts
    int kp_stride = 0;
    const double *p4 = nullptr;  // epipolar prior, or null
    const unsigned char *p4_has = nullptr;
    bool operator==(const FrameLaunch &o) const {
        return src == o.src && observs == o.observs && error == o.error && depth == o.depth && kp2d == o.kp2d &&
               xyz == o.xyz && obs_uv == o.obs_uv && kf_pose == o.kf_pose && kf_intr == o.kf_intr &&
               kf_bounds == o.kf_bounds && obs_ptr == o.obs_ptr && vis == o.vis && obs_kf == o.obs_kf &&
               kf_packed == o.kf_packed && kf_ptr == o.kf_ptr && nKF == o.nKF && obs_kf_bytes == o.obs_kf_bytes &&
               nnz == o.nnz && kf_slice_max == o.kf_slice_max && kf_bucket == o.kf_bucket && ucam == o.ucam &&
               memcmp(cam8, o.cam8, sizeof(cam8)) == 0 && map == o.map && kp_tab == o.kp_tab &&
               kp_stride == o.kp_stride && p4 == o.p4 && p4_has == o.p4_has;
    }
};

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

// one set of device-resident inputs of a frames batch.  Two sets exist so that lccrf_frames_submit_* can upload
// step i+1 on the copy stream while step i computes (the graph of a slot reads that slot's buffers).
struct FrameInputs {
    // direct inputs (Tracking.cc:1849-1870 vectors)
    float *observs = nullptr, *error = nullptr, *depth = nullptr;
    float *kp2d = nullptr;  // [NT*2], every source
    // map snapshot
    float *xyz = nullptr, *obs_uv = nullptr, *kf_pose = nullptr, *kf_intr = nullptr, *kf_bounds = nullptr;
    int *obs_ptr = nullptr;
    void *obs_kf = nullptr;  // int32 or uint16 keyframe indices, or {keyframe, feature index} pairs of them
    void *kf_packed = nullptr;
    int *kf_ptr = nullptr;   // [B+1] keyframe slice of each problem (optional)
    int nKF_cap = 0;
    long long nnz_cap = 0;   // obs_kf (and obs_uv, when allocated) hold this many observations
    // frame points named by ids of a device-resident map
    int *vis = nullptr;      // [NT] map point ids
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
    // label-application lists delivered by the pipelined submissions (lccrf_frames_set_partition_outputs)
    const int *part_fid = nullptr;
    int *part_dyn_ptr = nullptr, *part_dyn = nullptr, *part_stat_ptr = nullptr, *part_stat = nullptr;
    bool have_inputs = false;
    FrameLaunch launch;        // launch arguments of the next run as the last upload left them (kp_tab: at the run)
    FrameLaunch graph_launch;  // launch arguments `graph` was captured for
    GraphReplay graph;
    cudaEvent_t up_done = nullptr, run_done = nullptr, out_done = nullptr;
    int *h_status = nullptr;  // pinned copy of the device status word taken after this slot's run
    bool in_flight = false;
};

// the label-application lists in lccrf_frames::part
struct PartitionDev {
    int *dyn_ptr, *stat_ptr, *dyn, *stat;  // [B+1], [B+1] (right behind dyn_ptr), [NT], [NT]
};

}  // namespace

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
};

// entry points that read or replace what a pipelined submission still uses
static int frames_check_idle(const lccrf_frames *fr) {
    for (const FrameInputs &in : fr->in)
        if (in.in_flight)
            return fail(LCCRF_ERR_STATE, "a pipelined submission is in flight: call lccrf_frames_wait for both slots first");
    return LCCRF_OK;
}

// (Re)allocate a buffer of input set `in`, filled on stream `st`.  Input buffers are stream-ordered allocations of
// ctx->stream, but the pipelined submit path fills them on the copy stream: after an allocation the copy stream is
// ordered behind ctx->stream, so that a block the pool recycled from work still running there (the other slot's step)
// is not overwritten early.  Steady state allocates nothing.
template <typename T>
static int slot_alloc(Ctx *ctx, FrameInputs &in, cudaStream_t st, T *&p, size_t bytes) {
    dev_free(ctx, p);
    p = nullptr;
    LCCRF_TRY(dev_alloc(ctx, (void **)&p, bytes));
    if (st == ctx->stream || !in.up_done) return LCCRF_OK;
    LCCRF_CUDA(cudaEventRecord(in.up_done, ctx->stream));
    LCCRF_CUDA(cudaStreamWaitEvent(st, in.up_done, 0));
    return LCCRF_OK;
}

// optional keyframe slices kf_ptr [B+1] of the problems: they must span [0, nKF]; *slice_max = the largest (0 without)
static int check_kf_ptr(const int *kf_ptr, int B, int nKF, int *slice_max) {
    *slice_max = 0;
    if (!kf_ptr) return LCCRF_OK;
    if (kf_ptr[0] != 0 || kf_ptr[B] != nKF) return fail(LCCRF_ERR_ARG, "kf_ptr must span [0, number of keyframes]");
    for (int i = 0; i < B; i++) {
        if (kf_ptr[i + 1] < kf_ptr[i]) return fail(LCCRF_ERR_ARG, "kf_ptr must be non-decreasing");
        *slice_max = std::max(*slice_max, kf_ptr[i + 1] - kf_ptr[i]);
    }
    return LCCRF_OK;
}

// the end of every upload: the frame's keypoints, the epipolar prior registered with lccrf_frames_set_prior, and the
// launch key k of the next run
static int frames_upload_finish(lccrf_frames *fr, FrameInputs &in, cudaStream_t st, const float *kp2d, FrameLaunch k) {
    Ctx *ctx = fr->ctx;
    const size_t n = (size_t)fr->b.NT;
    if (!in.kp2d) LCCRF_TRY(slot_alloc(ctx, in, st, in.kp2d, (n ? n : 1) * 8));
    if (n) LCCRF_CUDA(cudaMemcpyAsync(in.kp2d, kp2d, n * 8, cudaMemcpyHostToDevice, st));
    k.kp2d = in.kp2d;
    if (in.h_p4 && n) {
        if (!in.p4) {
            LCCRF_TRY(slot_alloc(ctx, in, st, in.p4, n * sizeof(double)));
            LCCRF_TRY(slot_alloc(ctx, in, st, in.p4_has, (size_t)fr->b.B));
        }
        k.p4 = in.p4;
        LCCRF_CUDA(cudaMemcpyAsync(in.p4, in.h_p4, n * sizeof(double), cudaMemcpyHostToDevice, st));
        if (in.h_p4_has) {
            k.p4_has = in.p4_has;
            LCCRF_CUDA(cudaMemcpyAsync(in.p4_has, in.h_p4_has, (size_t)fr->b.B, cudaMemcpyHostToDevice, st));
        }
    }
    in.launch = k;
    in.have_inputs = true;
    return LCCRF_OK;
}

// upload the direct per-frame vectors of one step into input set `in` on stream `st`
static int frames_upload_direct(lccrf_frames *fr, FrameInputs &in, cudaStream_t st, const float *observs,
                                const float *error, const float *depth, const float *kp2d) {
    Ctx *ctx = fr->ctx;
    const size_t n = (size_t)fr->b.NT, m = n ? n : 1;
    if (n && (!observs || !error || !depth || !kp2d)) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (!in.observs) {
        LCCRF_TRY(slot_alloc(ctx, in, st, in.observs, m * 4));
        LCCRF_TRY(slot_alloc(ctx, in, st, in.error, m * 4));
        LCCRF_TRY(slot_alloc(ctx, in, st, in.depth, m * 4));
    }
    if (n) {
        LCCRF_CUDA(cudaMemcpyAsync(in.observs, observs, n * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.error, error, n * 4, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.depth, depth, n * 4, cudaMemcpyHostToDevice, st));
    }
    FrameLaunch k;
    k.src = FrameSource::kDirect;
    k.observs = in.observs;
    k.error = in.error;
    k.depth = in.depth;
    return frames_upload_finish(fr, in, st, kp2d, k);
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
    FrameLaunch k;
    k.src = indexed ? FrameSource::kSnapshotIndexed : FrameSource::kSnapshot;
    LCCRF_TRY(check_kf_ptr(kf_ptr, fr->b.B, nKF, &k.kf_slice_max));
    k.ucam = nnz > 0 && uniform_camera(kf_intr, kf_bounds, nKF, k.cam8);
    if (nnz > in.nnz_cap || !in.obs_kf || (!indexed && !in.obs_uv)) {
        in.nnz_cap = std::max(nnz, in.nnz_cap);
        const size_t bytes = (size_t)(in.nnz_cap ? in.nnz_cap : 1) * 8;  // obs_kf: up to an int32 {kf, fid} pair
        LCCRF_TRY(slot_alloc(ctx, in, st, in.obs_kf, bytes));
        dev_free(ctx, in.obs_uv);
        in.obs_uv = nullptr;
        if (!indexed) LCCRF_TRY(slot_alloc(ctx, in, st, in.obs_uv, bytes));
    }
    if (nKF > in.nKF_cap || !in.kf_pose) {
        const size_t n = (size_t)(nKF ? nKF : 1);
        LCCRF_TRY(slot_alloc(ctx, in, st, in.kf_pose, n * 48));
        LCCRF_TRY(slot_alloc(ctx, in, st, in.kf_intr, n * 16));
        LCCRF_TRY(slot_alloc(ctx, in, st, in.kf_bounds, n * 16));
        LCCRF_TRY(slot_alloc(ctx, in, st, in.kf_packed, n * 80));
        in.nKF_cap = nKF;
    }
    if (!in.xyz) {
        LCCRF_TRY(slot_alloc(ctx, in, st, in.xyz, (size_t)(NT ? NT : 1) * 12));
        LCCRF_TRY(slot_alloc(ctx, in, st, in.obs_ptr, (size_t)(NT + 1) * 4));
    }
    if (kf_ptr && !in.kf_ptr) LCCRF_TRY(slot_alloc(ctx, in, st, in.kf_ptr, (size_t)(fr->b.B + 1) * 4));
    k.xyz = in.xyz;
    k.obs_ptr = in.obs_ptr;
    k.obs_kf = in.obs_kf;
    k.obs_uv = indexed ? nullptr : in.obs_uv;
    k.kf_pose = in.kf_pose;
    k.kf_intr = in.kf_intr;
    k.kf_bounds = in.kf_bounds;
    k.kf_packed = in.kf_packed;
    k.kf_ptr = kf_ptr ? in.kf_ptr : nullptr;
    k.nKF = nKF;
    k.nnz = nnz;
    k.obs_kf_bytes = obs_kf_bytes;
    if (kf_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.kf_ptr, kf_ptr, (size_t)(fr->b.B + 1) * 4, cudaMemcpyHostToDevice, st));
    if (NT > 0) {
        LCCRF_CUDA(cudaMemcpyAsync(in.xyz, xyz, (size_t)NT * 12, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.obs_ptr, obs_ptr, (size_t)(NT + 1) * 4, cudaMemcpyHostToDevice, st));
    }
    if (nnz > 0) {
        LCCRF_CUDA(cudaMemcpyAsync(in.obs_kf, obs_kf, (size_t)nnz * obs_kf_bytes * (indexed ? 2 : 1), cudaMemcpyHostToDevice, st));
        if (!indexed) LCCRF_CUDA(cudaMemcpyAsync(in.obs_uv, obs_uv, (size_t)nnz * 8, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kf_pose, kf_pose, (size_t)nKF * 48, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kf_intr, kf_intr, (size_t)nKF * 16, cudaMemcpyHostToDevice, st));
        LCCRF_CUDA(cudaMemcpyAsync(in.kf_bounds, kf_bounds, (size_t)nKF * 16, cudaMemcpyHostToDevice, st));
    }
    return frames_upload_finish(fr, in, st, kp2d, k);
}

// frame points named by ids of the resident map (+ the step's map delta) into input set `in` on stream `st`
static int frames_upload_visible(lccrf_frames *fr, FrameInputs &in, cudaStream_t st, lccrf_map *map, const lccrf_map_delta *delta,
                                 const int *point_id, const float *kp2d, const int *kf_ptr) {
    Ctx *ctx = fr->ctx;
    if (!map || !map->m) return fail(LCCRF_ERR_ARG, "map is NULL");
    DevMap *m = map->m;
    if (m->ctx != ctx) return fail(LCCRF_ERR_ARG, "map and frames belong to different contexts");
    const int NT = fr->b.NT, B = fr->b.B;
    if (NT > 0 && (!point_id || !kp2d)) return fail(LCCRF_ERR_ARG, "NULL argument");
    const bool pipelined = st != ctx->stream;
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
        // host-side bookkeeping + capacity growth.  Pipelined: stream-ordered on the MAP's stream behind the last access
        // of the context's stream (an array that moves is freed there, and the previous step's unary may still read it)
        LCCRF_TRY(pipelined ? map_begin_async_mut(m) : map_begin_main_access(m));
        MapStreamScope on_map_stream(m, pipelined);
        LCCRF_TRY(map_prepare(m, *delta));
        LCCRF_TRY(delta_grow_points(m, *delta));
    }
    if (m->n_kf <= 0 && NT > 0) return fail(LCCRF_ERR_STATE, "the map has no keyframes");
    FrameLaunch k;
    k.src = FrameSource::kVisible;
    LCCRF_TRY(check_kf_ptr(kf_ptr, B, m->n_kf, &k.kf_slice_max));
    k.ucam = m->cam_set && m->ucam;
    if (k.ucam) memcpy(k.cam8, m->cam8, sizeof(k.cam8));
    k.kf_bucket = (m->n_kf + 127) / 128 * 128;
    if (!in.vis) LCCRF_TRY(slot_alloc(ctx, in, st, in.vis, (size_t)(NT ? NT : 1) * 4));
    if (kf_ptr && !in.kf_ptr) LCCRF_TRY(slot_alloc(ctx, in, st, in.kf_ptr, (size_t)(B + 1) * 4));
    k.vis = in.vis;
    k.kf_ptr = kf_ptr ? in.kf_ptr : nullptr;
    k.map = m;
    in.has_delta = false;
    if (delta) {
        if (pipelined) {
            LCCRF_TRY(delta_stage(*delta, m->kp_stride, true, (char *)in.stage, st, &in.delta));
            in.has_delta = true;  // applied on the map's stream once the upload has landed (frames_run_slot)
        } else {
            DeltaDev dd;
            LCCRF_TRY(delta_stage(*delta, m->kp_stride, false, (char *)in.stage, st, &dd));
            LCCRF_TRY(map_apply_dev(m, dd, delta->kf_count > 0 ? delta->kf_keypoints : nullptr));
        }
    }
    if (kf_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.kf_ptr, kf_ptr, (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, st));
    if (NT > 0) LCCRF_CUDA(cudaMemcpyAsync(in.vis, point_id, (size_t)NT * 4, cudaMemcpyHostToDevice, st));
    return frames_upload_finish(fr, in, st, kp2d, k);
}

static int frames_enqueue(lccrf_frames *fr, const FrameLaunch &k) {
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
        LCCRF_TRY(feat_div2(ctx, fr->feat2, k.kp2d, 2, prm.point2d_stdev, k.kp2d + 1, 2, prm.point2d_stdev, NT));
        LCCRF_TRY(lattice_set_build(ctx, b, b.lat[1], fr->feat2));
        LCCRF_TRY(potts_norm(ctx, b, b.lat[1]));
    }
    const float *cam8 = k.ucam ? k.cam8 : nullptr;
    if (k.src == FrameSource::kVisible) {
        LCCRF_TRY(unary_map_points_visible(ctx, NT, k.vis, k.map->d_hdr, k.kf_bucket, fr->observs, fr->error, fr->depth,
                                           b.prob_ptr, k.kf_ptr, b.B, k.kf_slice_max, cam8));
        LCCRF_TRY(map_end_main_access(k.map));  // the map may change from here on (the next step's delta, on the map's stream)
    } else if (k.src != FrameSource::kDirect) {
        LCCRF_TRY(unary_pack_kf(ctx, k.kf_packed, k.kf_pose, k.kf_intr, k.kf_bounds, k.nKF));
        LCCRF_TRY(unary_map_points_packed(ctx, NT, k.nKF, k.xyz, k.obs_ptr, k.obs_kf, k.obs_kf_bytes, k.obs_uv, k.kf_packed,
                                          fr->observs, fr->error, fr->depth, b.prob_ptr, k.kf_ptr, b.B, k.kf_slice_max,
                                          cam8, k.kp_tab, k.kp_stride));
    }
    const bool direct = k.src == FrameSource::kDirect;
    const float *observs = direct ? k.observs : fr->observs, *error = direct ? k.error : fr->error,
                *depth = direct ? k.depth : fr->depth;
    // RroughClassify -> setUnaryEnergyFromLabel   (Tracking.cc:1871,1921)
    LCCRF_TRY(unary_classify(ctx, NT, observs, error, depth, k.p4, prm, fr->label, k.p4_has, b.prob_ptr, b.B));
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

// Run the batch from input set `in` on ctx->stream, with CUDA-graph replay when enabled.  upload_stream: the stream
// the pipelined submissions uploaded the inputs on (null for the synchronous path).
static int frames_run_slot(lccrf_frames *fr, FrameInputs &in, cudaStream_t upload_stream) {
    Ctx *ctx = fr->ctx;
    if (!in.have_inputs) return fail(LCCRF_ERR_STATE, "frames_run before set_inputs");
    FrameLaunch k = in.launch;
    if (k.src == FrameSource::kSnapshotIndexed) {  // the table moves when keyframes are inserted
        k.kp_tab = fr->kp_tab;
        k.kp_stride = fr->kp_stride;
    }
    if (!(k == in.graph_launch)) {
        graph_drop(in.graph);
        in.graph_launch = k;
    }
    // behind the key comparison: a run that starts a new shape captures nothing and needs no synchronisation
    if (upload_stream && graph_will_capture(ctx, in.graph)) {
        // the capture pass synchronises; make sure the upload has landed first
        LCCRF_CUDA(cudaStreamSynchronize(upload_stream));
    }
    if (in.has_delta) {
        // this step's map changes: plain launches on the map's own stream, behind the upload and behind the previous
        // step's unary -- they run beside that step's lattice builds and mean-field iterations
        in.has_delta = false;
        LCCRF_CUDA(cudaStreamWaitEvent(k.map->mstream, in.up_done, 0));
        {
            MapStreamScope on_map_stream(k.map);
            LCCRF_TRY(map_apply_dev(k.map, in.delta, nullptr));
        }
        LCCRF_TRY(map_end_async_mut(k.map));
    }
    if (k.src == FrameSource::kVisible) LCCRF_TRY(map_begin_main_access(k.map));
    LCCRF_TRY(graph_run(ctx, in.graph, [&] { return frames_enqueue(fr, k); }));
    fr->ran = true;
    return LCCRF_OK;
}

// label application (Tracking.cc:1945-1955): stable partition of the batch's MAP labels on ctx->stream into the
// workspace fr->part; fid (host, [NT] or null) names the points in the lists
static int frames_partition_enqueue(lccrf_frames *fr, const int *fid, PartitionDev *out) {
    Ctx *ctx = fr->ctx;
    const int NT = fr->b.NT, B = fr->b.B;
    const size_t nB = (size_t)(B + 1), nT = (size_t)(NT > 0 ? NT : 1);
    if (!fr->part)
        LCCRF_TRY(dev_alloc(ctx, (void **)&fr->part, (2 * nB + 3 * nT) * sizeof(int) + label_partition_scratch_bytes(NT)));
    PartitionDev d;
    d.dyn_ptr = fr->part;
    d.stat_ptr = d.dyn_ptr + nB;
    d.dyn = d.stat_ptr + nB;
    d.stat = d.dyn + nT;
    int *d_fid = d.stat + nT, *d_scratch = d_fid + nT;
    if (fid && NT) LCCRF_CUDA(cudaMemcpyAsync(d_fid, fid, (size_t)NT * 4, cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_TRY(label_partition(ctx, fr->b.map, NT, fr->b.prob_ptr, B, fid ? d_fid : nullptr, d_scratch, d.dyn_ptr, d.dyn,
                              d.stat_ptr, d.stat));
    *out = d;
    return LCCRF_OK;
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
    LCCRF_TRY(frames_run_slot(fr, in, ctx->copy_stream));
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
        // label application of THIS submission, before the other slot's run reuses the labels
        const size_t nB = (size_t)(fr->b.B + 1), NT = (size_t)fr->b.NT;
        PartitionDev d;
        LCCRF_TRY(frames_partition_enqueue(fr, in.part_fid, &d));
        cudaStream_t st = ctx->stream;
        if (in.part_dyn_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.part_dyn_ptr, d.dyn_ptr, nB * 4, cudaMemcpyDeviceToHost, st));
        if (in.part_stat_ptr) LCCRF_CUDA(cudaMemcpyAsync(in.part_stat_ptr, d.stat_ptr, nB * 4, cudaMemcpyDeviceToHost, st));
        if (in.part_dyn && NT) LCCRF_CUDA(cudaMemcpyAsync(in.part_dyn, d.dyn, NT * 4, cudaMemcpyDeviceToHost, st));
        if (in.part_stat && NT) LCCRF_CUDA(cudaMemcpyAsync(in.part_stat, d.stat, NT * 4, cudaMemcpyDeviceToHost, st));
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

extern "C" {

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

int lccrf_frames_set_map_inputs_indexed(lccrf_frames *fr, const float *xyz, const int *obs_ptr, const void *obs_ref,
                                        int index_bytes, int nKF, const float *kf_pose, const float *kf_intr,
                                        const float *kf_bounds, const float *kp2d, const int *kf_ptr) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    return frames_upload_map(fr, fr->in[0], fr->ctx->stream, xyz, obs_ptr, obs_ref, index_bytes, nullptr, nKF, kf_pose,
                             kf_intr, kf_bounds, kp2d, kf_ptr, true);
}

int lccrf_frames_set_visible(lccrf_frames *fr, lccrf_map *map, const lccrf_map_delta *delta, const int *point_id,
                             const float *kp2d, const int *kf_ptr) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    LCCRF_TRY(frames_check_idle(fr));
    LCCRF_TRY(frames_upload_visible(fr, fr->in[0], fr->ctx->stream, map, delta, point_id, kp2d, kf_ptr));
    // the host arrays (delta included) are free on return
    LCCRF_CUDA(cudaStreamSynchronize(fr->ctx->stream));
    return LCCRF_OK;
}

int lccrf_frames_set_prior(lccrf_frames *fr, int slot, const double *p4, const unsigned char *has_prior) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (slot < 0 || slot > 1) return fail(LCCRF_ERR_ARG, "slot must be 0 or 1");
    if (!p4 && has_prior) return fail(LCCRF_ERR_ARG, "has_prior without p4");
    fr->in[slot].h_p4 = p4;
    fr->in[slot].h_p4_has = has_prior;
    return LCCRF_OK;
}

// ---- resident keyframe keypoints (indexed observations) ----
int lccrf_frames_set_keyframe_keypoints(lccrf_frames *fr, int kf_first, int kf_count, int stride, const float *kp_uv) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (kf_first < 0 || kf_count < 0 || stride <= 0) return fail(LCCRF_ERR_ARG, "bad keyframe range or stride");
    if (kf_count > 0 && !kp_uv) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (fr->kp_tab && stride != fr->kp_stride) return fail(LCCRF_ERR_ARG, "stride differs from the resident table's");
    LCCRF_TRY(frames_check_idle(fr));
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const long long need = (long long)kf_first + kf_count;
    if (need > 0x7fffffffLL) return fail(LCCRF_ERR_ARG, "too many keyframes");
    if (!fr->kp_tab || need > fr->kp_cap) {  // the table moves: the slots' next runs see a new launch key
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
    }
    if (kf_count > 0)
        LCCRF_CUDA(cudaMemcpyAsync(fr->kp_tab + (size_t)kf_first * stride * 2, kp_uv, (size_t)kf_count * stride * 8,
                                   cudaMemcpyHostToDevice, ctx->stream));
    // rare call (keyframe insertion): synchronise so that the host buffer is free on return and the copy stream of
    // the pipelined submissions sees the table
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return LCCRF_OK;
}

int lccrf_frames_run(lccrf_frames *fr) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    LCCRF_CUDA(cudaSetDevice(fr->ctx->device));
    fr->last_slot = 0;
    return frames_run_slot(fr, fr->in[0], nullptr);
}

int lccrf_frames_get_outputs(lccrf_frames *fr, short *map, float *prob) {
    if (!fr) return fail(LCCRF_ERR_ARG, "frames is NULL");
    if (!fr->ran) return fail(LCCRF_ERR_STATE, "frames_get_outputs before frames_run");
    LCCRF_TRY(frames_check_idle(fr));
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)fr->b.NT;
    if (n && map) LCCRF_CUDA(cudaMemcpyAsync(map, fr->b.map, n * 2, cudaMemcpyDeviceToHost, ctx->stream));
    if (n && prob) LCCRF_CUDA(cudaMemcpyAsync(prob, fr->b.cur, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return check_status(ctx);
}

int lccrf_frames_submit(lccrf_frames *fr, int slot, const float *observs, const float *error, const float *depth,
                        const float *kp2d, short *map_out, float *prob_out) {
    FrameInputs *in = nullptr;
    LCCRF_TRY(frames_submit_prologue(fr, slot, &in));
    LCCRF_TRY(frames_upload_direct(fr, *in, fr->ctx->copy_stream, observs, error, depth, kp2d));
    return frames_submit_epilogue(fr, slot, *in, map_out, prob_out);
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
    LCCRF_TRY(frames_check_idle(fr));
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)fr->b.NT;
    cudaStream_t st = ctx->stream;
    const FrameInputs &in = fr->in[fr->last_slot];
    const bool direct = in.launch.src == FrameSource::kDirect;
    const float *d_obs = direct ? in.observs : fr->observs, *d_err = direct ? in.error : fr->error,
                *d_dep = direct ? in.depth : fr->depth;
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
    LCCRF_TRY(frames_check_idle(fr));
    Ctx *ctx = fr->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const int NT = fr->b.NT, B = fr->b.B;
    const size_t nB = (size_t)(B + 1);
    PartitionDev d;
    LCCRF_TRY(frames_partition_enqueue(fr, fid, &d));
    cudaStream_t st = ctx->stream;
    std::vector<int> hp(2 * nB);
    LCCRF_CUDA(cudaMemcpyAsync(hp.data(), d.dyn_ptr, 2 * nB * sizeof(int), cudaMemcpyDeviceToHost, st));
    LCCRF_CUDA(cudaStreamSynchronize(st));
    const int n_dyn = hp[B], n_stat = hp[nB + B];
    if (n_dyn < 0 || n_stat < 0 || n_dyn + n_stat != NT) return fail(LCCRF_ERR_STATE, "label partition is inconsistent");
    if (dyn_ptr) memcpy(dyn_ptr, hp.data(), nB * sizeof(int));
    if (stat_ptr) memcpy(stat_ptr, hp.data() + nB, nB * sizeof(int));
    if (dyn_list && n_dyn) LCCRF_CUDA(cudaMemcpyAsync(dyn_list, d.dyn, (size_t)n_dyn * 4, cudaMemcpyDeviceToHost, st));
    if (stat_list && n_stat) LCCRF_CUDA(cudaMemcpyAsync(stat_list, d.stat, (size_t)n_stat * 4, cudaMemcpyDeviceToHost, st));
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
    const FrameLaunch &k = fr->in[fr->last_slot].launch;
    long long nnz = k.nnz;
    int nKF = k.nKF;
    if (k.src == FrameSource::kVisible) {  // observations of the visible points: counted on the device
        nKF = k.map->n_kf;
        nnz = 0;
        if (fr->b.NT > 0) {
            Ctx *ctx = fr->ctx;
            int *d_cnt = nullptr;
            LCCRF_TRY(dev_alloc(ctx, (void **)&d_cnt, (size_t)fr->b.NT * 4));
            int rc = map_export_dev(k.map, fr->b.NT, k.vis, d_cnt);
            std::vector<int> cnt((size_t)fr->b.NT);
            if (rc == LCCRF_OK) {
                cudaError_t e = cudaMemcpyAsync(cnt.data(), d_cnt, cnt.size() * 4, cudaMemcpyDeviceToHost, ctx->stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
                if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, cudaGetErrorString(e));
            }
            dev_free(ctx, d_cnt);
            LCCRF_TRY(rc);
            for (int c : cnt) nnz += c;
        }
    }
    if (k.src != FrameSource::kDirect) u = (double)nnz * 12 + (double)fr->b.NT * 24 + (double)nKF * 80;
    if (total) *total = tot + u;
    if (per_iteration) *per_iteration = it_tot;
    if (unary) *unary = u;
    return LCCRF_OK;
}

}  // extern "C"
