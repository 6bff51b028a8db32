// engine.cuh -- internal data model of liblccrf: a *batch* of B independent CRF problems whose
// points are concatenated (problem b owns points [prob_ptr[b], prob_ptr[b+1])).  A single
// DenseCRF object is a batch with B == 1.  Everything lives in HBM; the layouts are chosen for
// coalesced streaming (see DESIGN.md "Data layout").
#pragma once

#include <cstddef>
#include <functional>
#include <vector>

#include "common.cuh"

namespace lccrf {

struct Ctx;

// One pairwise kernel (one permutohedral lattice per problem) across the whole batch.
struct LatticeSet {
    int d = 0, D = 0;
    float w = 0.f;      // Potts weight w_ (pairwise3d.h:17)
    float alpha = 0.f;  // 1/(1+2^-d) (permutohedral_cpu.h:681)
    int NT = 0, B = 0;
    int Vcap = 0;       // capacity of the per-vertex arrays: (NT + B) * D worst case
    // per (point, remainder), tight point-major [NT*D]: GLOBAL vertex id (= vbase[b] + reference id)
    int *offset = nullptr;
    float *bary = nullptr;
    // per vertex
    int2 *nbr = nullptr;        // [D][Vcap] {n1,n2} global ids, -1 = absent   (permutohedral_cpu.h:418-419)
    int *vert_slot = nullptr;   // [Vcap] hash slot of each vertex (build only)
    int *vert_prob = nullptr;   // [Vcap] owning problem
    int *vbase = nullptr;       // [B+1] first global vertex id of each problem; vbase[B] = V_total
    int *tab_base = nullptr;    // [B+1] first hash slot of each problem's open-addressing region (build only)
    long long tab_slots = 0;
    float *norm = nullptr;      // [NT] 1/(filter(1)+1e-20)   (pairwise3d.h:22-27)
    // vertex-sorted view for the splat (csr.cu): row v = entries [row_ptr[v], row_ptr[v+1]) in point order
    int *row_ptr = nullptr;     // [Vcap+2]
    int2 *csr_ent = nullptr;    // [NT*D] {global point index, bary bits}
    int csr_chunks = 0;
    int *chunk_prob = nullptr, *chunk_s0 = nullptr, *chunk_s1 = nullptr, *prob_chunk0 = nullptr;
    long long *chunk_tbl = nullptr;
    int *csr_tbl = nullptr, *scan_tot = nullptr;
    // long rows (>= kLongRow entries; filled by csr_build) and their chunks of kScanChunk entries (filter.cu: speculative scan)
    int *row_list_long = nullptr;   // [max_long] vertex ids
    int *row_counts = nullptr;      // [8] device: #long rows, #chunks, #pieces, compose ticket, 4 walk diagnostics
    int *long_chunk0 = nullptr;     // [max_long+1] first chunk of each long row
    void *chunk_desc = nullptr;     // [max_chunks] int4 {first entry, end entry, first chunk of the row, long-list index}
    unsigned long long *chunk_sum = nullptr;  // [max_chunks*Lmax] {call tag, unordered fp32 chunk sum}: published and polled inside k_scan_compose
    void *chunk_rec = nullptr;      // [max_chunks*Lmax] ChunkRec (per filter call)
    int max_long = 0, max_chunks = 0;
    // pieces (diagnostic, lccrf_frames debug counters): first rows of the maximal runs of short rows that start in one kTileGranule granule
    int *piece_list = nullptr;      // [max_pieces]
    int max_pieces = 0;
    // tree splat (option "ordered_splat" = 0): fixed tiles of kTreeTile sorted entries
    int n_tiles = 0;
    int *tile_row0 = nullptr;       // [n_tiles+1] row that holds the first entry of each tile; [n_tiles] = V-1
    int *tile_own = nullptr;        // [n_tiles] != 0: the ordered short-row splat has rows to sum in this tile
    int2 *tile_info = nullptr;      // [n_tiles] {position of the first row start inside the tile or -1, row open at the tile's end or -1}
    float *tile_part = nullptr;     // [n_tiles*Lmax] sum of the tile's entries in front of its first row start
    // filter workspace
    float *valA = nullptr, *valB = nullptr;  // [Vcap*Lmax] blur ping-pong
    int Lmax = 0;
};

constexpr int kCsrChunkPoints = 4096;  // points per chunk of the parallel stable counting sort
constexpr int kLongRow = 1024;    // rows at least this long leave the staged lane-sequential kernel for the exact scan
constexpr int kScanChunk = 2048;  // entries per chunk of a long row
constexpr int kChunkRecBytes = 16 + 2 * 24 + 4 * (kScanChunk / 256) * 4;  // sizeof(ChunkRec) of filter.cu
constexpr int kTileGranule = 2048;  // entry granularity of the row pieces
constexpr int kTreeTile = 2048;     // entries per tile of the tree splat (filter.cu: k_splat_tree)

struct Batch {
    Ctx *ctx = nullptr;
    int B = 0, NT = 0, L = 0;
    std::vector<int> h_prob_ptr;  // host copy
    int *prob_ptr = nullptr;      // [B+1] device
    int maxN = 0;
    // blur of every filter call: true = k_blur_fused, one CTA per problem runs all D passes out of shared memory;
    // false = element-parallel passes (k_blur_bulk / k_blur_vec) over the vertices of all problems, one launch per pass
    bool fused_blur = false;
    std::vector<LatticeSet *> lat;  // K potentials
    float *unary = nullptr, *cur = nullptr, *next = nullptr, *tmp = nullptr;  // [NT*L]
    short *map = nullptr;                                                      // [NT]
};

// ------------------------------------------------------------------ context
struct Ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;  // uploads of the pipelined submit path (created on first use)
    cudaStream_t d2h_stream = nullptr;   // results of the pipelined submit path on their way to the host
    uint64_t launches = 0;
    // bumped whenever every captured graph goes stale: a scratch buffer moved (graphs hold raw pointers) or an option
    // changed the launch sequence (lccrf_ctx_set_option)
    uint64_t scratch_gen = 0;
    int opt_graphs = 1;
    int opt_fused = 1;
    // 1: splat sums every vertex row in point order (bit-identical to the reference's sequential loop);
    // 0: fixed-shape tree reduction per row (deterministic; marginals within the 1e-4 gate, not bit-identical)
    int opt_ordered_splat = 1;
    int opt_trace = 0;         // host-side phase times of the pipelined submissions on stderr
    int opt_bulk_blur = 1;     // element-parallel blur: stream neighbour pairs / own values with cp.async.bulk (0: plain loads)
    int opt_map_slack = 0;     // spare room (percent) behind every list of a bulk-loaded map; 0 = tight lists: the unary streams
                               // them 4% faster, and a list that grows later moves to the pool's tail once (map.cu)
    // per-kernel CUDA-event timing (option "profile"): every launch site is bracketed by two events
    int opt_profile = 0;
    struct ProfRec {
        const char *name;
        cudaEvent_t a, b;
    };
    std::vector<ProfRec> prof;
    // scratch for the lattice build (grown on demand, reused)
    struct Scratch {
        void *p = nullptr;
        size_t bytes = 0;
    };
    struct BuildScratch {  // lattice-build workspace; one set per concurrent branch
        Scratch hash_keys[3], hash_first, hash_id, ent_slot, ids_status;
        // hash_keys / hash_first are empty between builds (every build empties the slots it used); true while a build
        // that may have left slots in use is in progress or failed before its clear was enqueued
        bool hash_dirty = false;
    };
    BuildScratch bs[2];
    Scratch misc, feat, pinned_in, pinned_out, dev_io;
    // fork/join of independent launch sequences (the K lattices of one CRF): `stream` is the main branch,
    // `aux_stream` the second one.  Inside a graph capture the event edges become parallel graph branches.
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int opt_concurrent = 1;
    int branch = 0;  // 0 = launches go to `stream`, 1 = to `aux_stream` (see AuxScope)
    // second level, inside one filter call: the short-row splat of a lattice runs beside its long-row scan kernels
    // (disjoint vertex rows; one sub-stream per branch)
    cudaStream_t sub_stream[2] = {nullptr, nullptr};
    cudaEvent_t ev_sub_fork[2] = {nullptr, nullptr}, ev_sub_join[2] = {nullptr, nullptr};
    int opt_split_splat = 1;
    // kernels whose opt-in dynamic shared memory limit has been raised on this context's device (function attributes
    // are per device, and a context belongs to one host thread: no process-wide flag)
    std::vector<const void *> smem_attr_done;
    int *d_status = nullptr;   // device status word (key range overflow etc.)
    int *h_status = nullptr;   // pinned
};

int ctx_scratch(Ctx *ctx, Ctx::Scratch &s, size_t bytes, bool pinned = false);

// batches (api.cu).  batch_init sets fused_blur = B >= 2 || maxN <= kFusedBlurMaxN (the rule of lccrf_crf and lccrf_frames);
// a caller with another rule overwrites it before the first filter call.
constexpr int kFusedBlurMaxN = 32768;
int batch_init(Ctx *ctx, Batch &b, int B, const int *prob_ptr, int L, bool with_state);
void batch_release(Ctx *ctx, Batch &b);
// device status word: read (synchronises), clear, and turn the first error it holds into a return code
int check_status(Ctx *ctx);
int decode_status(int st);  // a status word -> error code (0: LCCRF_OK)

// CUDA-graph replay of a launch sequence whose shape repeats.  The first run of a shape launches plainly; the second
// runs once more uncaptured (every scratch buffer reaches its final size) and captures; later runs replay.  An object
// keeps the key of every launch argument that can change between its runs (RunShape, FrameLaunch) its graph was captured
// for and calls graph_drop when the next run's key differs, which makes that run the first of a new shape.
struct GraphReplay {
    cudaGraphExec_t exec = nullptr;
    int same_shape_runs = 0;  // runs since the launch sequence last changed shape (a graph is captured on the 2nd)
    uint64_t launches = 0;    // kernels one replay stands for
    uint64_t gen = 0;         // Ctx::scratch_gen at capture
};
void graph_drop(GraphReplay &g);
// true when the next graph_run will capture (it synchronises the context's stream)
bool graph_will_capture(const Ctx *ctx, const GraphReplay &g);
int graph_run(Ctx *ctx, GraphReplay &g, const std::function<int()> &enqueue);

// RAII bracket around one kernel launch: counts it and, in profile mode, times it with CUDA events
// recorded on the launching stream.
struct KernelScope {
    Ctx *c;
    int idx = -1;
    KernelScope(Ctx *ctx, const char *name) : c(ctx) {
        c->launches++;
        if (c->opt_profile) {
            Ctx::ProfRec r;
            r.name = name;
            if (cudaEventCreate(&r.a) == cudaSuccess && cudaEventCreate(&r.b) == cudaSuccess) {
                cudaEventRecord(r.a, c->stream);
                c->prof.push_back(r);
                idx = (int)c->prof.size() - 1;
            }
        }
    }
    ~KernelScope() {
        if (idx >= 0) cudaEventRecord(c->prof[idx].b, c->stream);
    }
};
#define LCCRF_KERNEL(ctx, name) ::lccrf::KernelScope _kscope_##__LINE__(ctx, name)
// fork: the aux branch starts after everything enqueued on the main branch so far; join: main waits for aux
bool ctx_concurrent(const Ctx *ctx);
int ctx_fork(Ctx *ctx);
int ctx_join(Ctx *ctx);
// launches inside the scope go to the aux branch (no-op when concurrency is off)
struct AuxScope {
    Ctx *c;
    cudaStream_t saved;
    bool on;
    explicit AuxScope(Ctx *ctx, bool enable = true) : c(ctx), saved(ctx->stream), on(enable && ctx_concurrent(ctx)) {
        if (on) {
            c->stream = c->aux_stream;
            c->branch = 1;
        }
    }
    ~AuxScope() {
        if (on) {
            c->stream = saved;
            c->branch = 0;
        }
    }
};
// raise a kernel's dynamic shared memory limit once per context (first launch; outside any graph capture because every
// captured sequence is run once uncaptured first)
template <typename Kernel>
inline int ensure_dyn_smem(Ctx *ctx, Kernel *kernel, int bytes) {
    const void *key = (const void *)kernel;
    for (const void *k : ctx->smem_attr_done)
        if (k == key) return LCCRF_OK;
    LCCRF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    ctx->smem_attr_done.push_back(key);
    return LCCRF_OK;
}

int dev_alloc(Ctx *ctx, void **p, size_t bytes, bool zero = false);
void dev_free(Ctx *ctx, void *p);

// ------------------------------------------------------------------ device-resident map (map.cu)
struct KfPack {  // one keyframe as the unary kernel reads it: rows of [Rcw|tcw], intrinsics, image bounds
    float4 r0, r1, r2, intr, bnd;
};

// The state Tracking::ComputeMapPointErrAndObserv dereferences (src/Tracking.cc:1803-1839), kept in HBM across frames:
// keyframes (pose, intrinsics, bounds, undistorted keypoints) and map points (world position + observation list).
// Observation lists live in one pool: point p owns pool entries [pt_start[p], pt_start[p] + pt_cnt[p]) out of a
// reserved run of pt_room[p]; a list that outgrows its run moves to the pool's tail with twice the room.
// Device-side directory of the map's arrays.  Kernels that a captured graph replays read the arrays through it, so the
// map may move its arrays (growth) or gain keyframes without invalidating the graph: only this block is rewritten.
struct MapHeader {
    const KfPack *kf_packed;
    const float *pt_xyz;
    const int *pt_start, *pt_cnt;
    const int *pool_kf;
    const float *pool_uv;
    int n_kf;
};

struct DevMap {
    Ctx *ctx = nullptr;
    MapHeader *d_hdr = nullptr;   // device copy, rewritten by map_publish()
    // The pipelined submissions apply a step's delta on the map's own stream, so that it overlaps the lattice builds and
    // mean-field iterations of the previous step (only that step's unary kernel reads the map):
    //   ev_touch  recorded on the context's stream behind its last access to the map (the unary of a frame batch --
    //             inside a captured graph as an external event-record node --, a synchronous mutation, an export)
    //   ev_mut    recorded on the map's stream behind the last asynchronous mutation
    // Asynchronous mutations wait for ev_touch; every access from the context's stream waits for ev_mut.
    cudaStream_t mstream = nullptr;
    cudaEvent_t ev_touch = nullptr, ev_mut = nullptr;
    int kp_stride = 0;
    // keyframes
    int kf_cap = 0, n_kf = 0;
    KfPack *kf_packed = nullptr;  // [kf_cap]
    float *kp_tab = nullptr;      // [kf_cap][kp_stride] float2   KeyFrame::mvKeysUn
    bool cam_set = false, ucam = true;
    float cam8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // map points
    int pt_cap = 0, n_pt = 0;
    float *pt_xyz = nullptr;      // [pt_cap*3]   MapPoint::mWorldPos
    int *pt_start = nullptr, *pt_cnt = nullptr, *pt_room = nullptr, *pt_stamp = nullptr;  // [pt_cap]
    // observation pool
    long long pool_cap = 0;
    int *pool_kf = nullptr;       // [pool_cap] keyframe index
    float *pool_uv = nullptr;     // [pool_cap] float2: the observed keypoint, resolved when the observation is added
    int *d_ctr = nullptr;         // device counters: [0] pool tail, [1] pool capacity, [2] live entries, [3] scratch
    int *h_ctr = nullptr;         // pinned snapshot of d_ctr
    cudaEvent_t ctr_ev = nullptr;
    bool ctr_pending = false;
    long long tail_seen = 0;      // last snapshot of the pool tail
    long long tail_unseen = 0;    // entries bulk loads added behind that snapshot (known exactly on the host)
    int epoch = 0;
};

// a lccrf_map_delta whose arrays are in device memory
struct DeltaDev {
    int kf_first = 0, kf_count = 0;
    const float *kf_pose = nullptr, *kf_intr = nullptr, *kf_bounds = nullptr, *kf_keypoints = nullptr;
    int n_pose = 0;
    const int *pose_kf = nullptr;
    const float *pose = nullptr;
    int n_xyz = 0;
    const int *xyz_id = nullptr;
    const float *xyz = nullptr;
    int n_erase = 0;
    const int *erase_pt = nullptr, *erase_kf = nullptr;
    int n_bad = 0;
    const int *bad_pt = nullptr;
    int n_add = 0;
    const int *add_pt = nullptr, *add_kf = nullptr, *add_fid = nullptr;
    std::vector<int> erase_seg, add_seg;  // host copies of the segment boundaries (empty = one segment)
};
// bytes of the staged arrays of a delta (every array 256-byte aligned); with_keypoints = false when the new keyframes'
// keypoints are copied straight from the host array
size_t delta_stage_bytes(const lccrf_map_delta &d, int kp_stride, bool with_keypoints);
// copy the delta's host arrays to `base` on stream st and describe them in `out`
int delta_stage(const lccrf_map_delta &d, int kp_stride, bool with_keypoints, char *base, cudaStream_t st, DeltaDev *out);
// explicit point ids name points the caller creates densely: raise the capacity to the largest id of the delta
int delta_grow_points(DevMap *m, const lccrf_map_delta &d);

int map_create(Ctx *ctx, int kp_stride, DevMap **out);
void map_destroy(DevMap *m);
// host-side bookkeeping of a delta before its kernels run: capacity growth (stream-ordered on ctx->stream), camera
// uniformity, keyframe / point counts.  Host arrays are only inspected where the header says so (kf_intr / kf_bounds).
int map_prepare(DevMap *m, const lccrf_map_delta &h);
// enqueue the kernels that apply a staged delta on ctx->stream (order: keyframes, poses, positions, erase, bad, add);
// kp_host != nullptr: the new keyframes' keypoints are copied straight from that host array (synchronous API)
int map_apply_dev(DevMap *m, const DeltaDev &d, const float *kp_host);
int map_bulk_observations(DevMap *m, int pt_first, int count, const int *obs_ptr_dev, const int *obs_ref_dev, long long nnz,
                          int slack_percent);
int map_publish(DevMap *m);  // rewrite the device-side directory after arrays moved / keyframes were added
// ordering between the context's stream and the map's own stream (see DevMap)
int map_begin_main_access(DevMap *m);   // context stream waits for the asynchronous mutations enqueued so far
int map_end_main_access(DevMap *m);     // ... and marks the end of its access (external record node while capturing)
int map_begin_async_mut(DevMap *m);     // map stream waits for the context stream's last access
int map_end_async_mut(DevMap *m);
// scope in which ctx->stream IS the map's stream: map.cu's launches, copies and allocations go there (no-op when
// enable is false)
struct MapStreamScope {
    Ctx *c;
    cudaStream_t saved;
    explicit MapStreamScope(DevMap *m, bool enable = true) : c(m->ctx), saved(m->ctx->stream) {
        if (enable) c->stream = m->mstream;
    }
    ~MapStreamScope() { c->stream = saved; }
};
int map_reserve_pool(DevMap *m, long long entries);
int map_reserve_points(DevMap *m, int n);
int map_bulk_reserve(DevMap *m, long long need);
int map_export_dev(DevMap *m, int n, const int *ids_dev, int *cnt_dev);
int map_export_entries_dev(DevMap *m, int n, const int *ids_dev, const int *ptr_dev, int *kf_dev, float *uv_dev, float *xyz_dev,
                           long long cap);
int map_counters(DevMap *m, long long *tail, long long *live);  // synchronises

// ------------------------------------------------------------------ stages (each enqueues kernels on ctx->stream)
// lattice build: features [NT*d] on device -> offset/bary/nbr/vbase (lattice_build.cu)
int lattice_set_create(Ctx *ctx, const Batch &b, int d, float w, int Lmax, LatticeSet **out);
void lattice_set_destroy(Ctx *ctx, LatticeSet *ls);
int lattice_set_build(Ctx *ctx, const Batch &b, LatticeSet *ls, const float *feat_dev);
int lattice_set_ensure_L(Ctx *ctx, LatticeSet *ls, int L);  // (re)allocate the filter workspace for L labels
// synchronises; slots of both branches' hash scratch that are not empty (0 between builds)
int build_scratch_in_use(Ctx *ctx, long long *slots);
// vertex-sorted CSR of a built lattice set (csr.cu)
int csr_create(Ctx *ctx, const Batch &b, LatticeSet *ls);
void csr_destroy(Ctx *ctx, LatticeSet *ls);
int csr_build(Ctx *ctx, const Batch &b, LatticeSet *ls);
// filter (filter.cu): out/in device [NT*L]
int filter_splat_blur(Ctx *ctx, const Batch &b, LatticeSet *ls, const float *in_dev, int L,
                      const float **values_out);
int filter_full(Ctx *ctx, const Batch &b, LatticeSet *ls, float *out_dev, const float *in_dev, int L);
int potts_norm(Ctx *ctx, const Batch &b, LatticeSet *ls);
// mean field (meanfield.cu)
// status (optional): a label outside [-1, L) sets 32 in the device status word and is read as unknown (u_energy)
int mf_unary_from_label(Ctx *ctx, float *unary, const short *label_dev, int NT, int L, float u_energy,
                        const float *n_en, const float *p_en, int *status = nullptr);
int mf_exp_and_normalize(Ctx *ctx, float *out, const float *in, int NT, int L, float scale, float relax);
int mf_start(Ctx *ctx, Batch &b);
int mf_step(Ctx *ctx, Batch &b, float relax);
int mf_build_map(Ctx *ctx, Batch &b);
int mf_negate(Ctx *ctx, float *out, const float *in, long long n);
// potts apply on arbitrary device arrays (plugin path): tmp = filter(in); out += (w*norm)*tmp
int mf_potts_apply(Ctx *ctx, const Batch &b, LatticeSet *ls, float *out, const float *in, float *tmp, int L);
// one potential of a mean-field step: next = (first ? -unary : next) + (w*norm)*filter(cur)
int mf_apply_fused(Ctx *ctx, const Batch &b, LatticeSet *ls, const float *cur, float *next, const float *unary,
                   bool first);
int launch_axpy_norm(Ctx *ctx, float *out, const float *tmp, const float *norm, float w, int NT, int L);
// fused point pass for L == 2: slice of every lattice + Potts apply + softmax (+ MAP) in one kernel
int mf_point_pass_l2(Ctx *ctx, Batch &b, const float *const *values, float relax, bool with_map);
// features (unary.cu)
int feat_div2(Ctx *ctx, float *feat, const float *a, int stride_a, float sa, const float *b, int stride_b,
              float sb, int N);
int feat_image(Ctx *ctx, float *feat, int W, int H, int F, float posdev, const void *img_dev, int is_u8,
               float featuredev);
// the features of feat_image for every image of a batch in one launch: image b is pixels [prob_ptr[b], prob_ptr[b+1]),
// width[b] pixels wide (device arrays [B+1] / [B]); img_dev [NT*(F-2)]
int feat_image_batch(Ctx *ctx, float *feat, int NT, int B, const int *prob_ptr, const int *width, int F, float posdev,
                     const void *img_dev, int is_u8, float featuredev);
int unary_pack_kf(Ctx *ctx, void *kf_packed /*nKF*80 B*/, const float *pose, const float *intr, const float *bnd, int nKF);
int unary_map_points_packed(Ctx *ctx, int N, int nKF, const float *xyz, const int *obs_ptr, const void *obs_kf,
                            int obs_kf_bytes, const float *obs_uv, const void *kf_packed, float *observs, float *error, float *depth,
                            const int *prob_ptr, const int *kf_ptr, int B, int kf_slice_max, const float *cam8,
                            const float *kp_tab, int kp_stride);
int unary_map_points_visible(Ctx *ctx, int N, const int *vis, const MapHeader *map_hdr, int n_kf_bucket, float *observs,
                             float *error, float *depth, const int *prob_ptr, const int *kf_ptr, int B, int kf_slice_max,
                             const float *cam8);
// kp_tab != nullptr: indexed observations -- obs_kf holds {keyframe, feature index} pairs (uint16 pairs when
// obs_kf_bytes == 2, int32 pairs when 4), obs_uv is unused and the observed keypoint is kp_tab[kf*kp_stride + fid]
int unary_map_points(Ctx *ctx, int N, const float *xyz, const int *obs_ptr, const int *obs_kf,
                     const float *obs_uv, int nKF, const float *kf_pose, const float *kf_intr,
                     const float *kf_bounds, float *observs, float *error, float *depth, const float *cam8);
// cam8 (host, 8 floats {fx fy cx cy, minx maxx miny maxy}) when every keyframe has the same intrinsics and image
// bounds, else nullptr; uniform_camera() decides from the host tables
bool uniform_camera(const float *kf_intr, const float *kf_bounds, int nKF, float *cam8);
// has_prior (optional, [B] bytes): problems whose flag is 0 take the no-prior branch (Tracking.cc:1994-1999)
int unary_classify(Ctx *ctx, int N, const float *observs, const float *error, const float *depth,
                   const double *p4, const lccrf_slam_params &prm, short *label, const unsigned char *has_prior = nullptr,
                   const int *prob_ptr = nullptr, int B = 0);

// label application (apply.cu): stable partition of MAP labels into moving / static lists; all device pointers
size_t label_partition_scratch_bytes(int NT);
int label_partition(Ctx *ctx, const short *map, int NT, const int *prob_ptr, int B, const int *fid, int *scratch,
                    int *dyn_ptr, int *dyn_list, int *stat_ptr, int *stat_list);

// frontend (frontend.cu): epipolar prior and brute-force Hamming kNN; all pointers are device pointers
int epipolar_prior(Ctx *ctx, int M, const int *fid1, const float *pt1, const float *pt2, const double *F9_host,
                   float u_gamma, float stdev_gamma, int nFeat, double *dis_by_fid, double *prob_by_fid, double *dis_m,
                   double *prob_m);
int bf_match_splits(int B, int max_nq, int max_nt);
int bf_match(Ctx *ctx, int B, int NQ, int max_nq, int max_nt, const int *q_ptr, const void *desc_q, const int *t_ptr,
             const void *desc_t, double ratio, int S, void *part /*[NQ*S] int4*/, int *match, int *knn /*[NQ*4] or null*/,
             int *n_match);

}  // namespace lccrf

// opaque handles of include/lccrf.h (their entry points are spread over api.cu, frames.cu and images.cu)
struct lccrf_ctx {
    lccrf::Ctx c;
};

struct lccrf_map {
    lccrf::DevMap *m = nullptr;
};
