// map.cu -- the device-resident SLAM map behind lccrf_map (include/lccrf.h).
//
// In the reference the observation lists (MapPoint::mObservations, include/MapPoint.h:115), the keyframe poses and the
// keyframe keypoints (KeyFrame::mvKeysUn, include/KeyFrame.h:164) are persistent map state: tracking only reads them
// (Tracking::ComputeMapPointErrAndObserv, src/Tracking.cc:1803-1839) and local mapping changes a little per keyframe
// (MapPoint::AddObservation / EraseObservation / SetBadFlag / SetWorldPos, src/MapPoint.cc:73-168; KeyFrame::SetPose,
// src/KeyFrame.cc:70).  Here the same state lives in HBM and the mutators are kernels, so that a frame costs the PCIe
// bus its list of visible points and the step's changes instead of the whole map.
//
// Layout: one observation pool (pool_kf int32, pool_uv float2 = the observed keypoint, resolved from the resident
// keyframe when the observation is added).  Point p owns pool[pt_start[p] .. +pt_cnt[p]) inside a run of pt_room[p]
// entries; a full run moves to the pool's tail with twice the room (amortised O(1) appends, order preserved).  The
// unary kernel (unary.cu, VIS) reads the lists in place.
#include <cstring>

#include "engine.cuh"

namespace lccrf {

namespace {

constexpr int kMinRoom = 4;
enum { kCtrTail = 0, kCtrCap = 1, kCtrLive = 2, kCtrBase = 3 };
// status bits (ctx->d_status): 1 lattice key range, 2 index out of range, 4 visible point without observations,
// 8 a point twice in one delta list, 16 observation pool exhausted
enum { kStIndex = 2, kStTwice = 8, kStPool = 16 };

__global__ void __launch_bounds__(kThreads)
k_map_set_kf(KfPack *__restrict__ tab, const float *__restrict__ pose, const float *__restrict__ intr,
             const float *__restrict__ bnd, int first, int count) {
    const int k = blockIdx.x * kThreads + threadIdx.x;
    if (k >= count) return;
    const float *P = pose + 12 * (size_t)k;
    KfPack o;
    o.r0 = make_float4(P[0], P[1], P[2], P[3]);
    o.r1 = make_float4(P[4], P[5], P[6], P[7]);
    o.r2 = make_float4(P[8], P[9], P[10], P[11]);
    o.intr = make_float4(intr[4 * k], intr[4 * k + 1], intr[4 * k + 2], intr[4 * k + 3]);
    o.bnd = make_float4(bnd[4 * k], bnd[4 * k + 1], bnd[4 * k + 2], bnd[4 * k + 3]);
    tab[first + k] = o;
}

__global__ void __launch_bounds__(kThreads)
k_map_set_pose(KfPack *__restrict__ tab, const int *__restrict__ ids, const float *__restrict__ pose, int n, int n_kf,
               int *__restrict__ status) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int k = ids ? __ldg(ids + i) : i;
    if ((unsigned)k >= (unsigned)n_kf) {
        atomicOr(status, kStIndex);
        return;
    }
    const float *P = pose + 12 * (size_t)i;
    tab[k].r0 = make_float4(P[0], P[1], P[2], P[3]);
    tab[k].r1 = make_float4(P[4], P[5], P[6], P[7]);
    tab[k].r2 = make_float4(P[8], P[9], P[10], P[11]);
}

__global__ void __launch_bounds__(kThreads)
k_map_set_xyz(float *__restrict__ pt_xyz, const int *__restrict__ ids, const float *__restrict__ xyz, int n, int pt_cap,
              int *__restrict__ status) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int p = ids ? __ldg(ids + i) : i;
    if ((unsigned)p >= (unsigned)pt_cap) {
        atomicOr(status, kStIndex);
        return;
    }
    pt_xyz[3 * (size_t)p] = xyz[3 * (size_t)i];
    pt_xyz[3 * (size_t)p + 1] = xyz[3 * (size_t)i + 1];
    pt_xyz[3 * (size_t)p + 2] = xyz[3 * (size_t)i + 2];
}

struct PoolArgs {
    int *pt_start, *pt_cnt, *pt_room, *pt_stamp;
    int *pool_kf;
    float2 *pool_uv;
    int *ctr;
    int *status;
    const float2 *kp_tab;
    int kp_stride, n_kf, pt_cap, stamp;
};

// a point may be named once per list and delta: the second thread that stamps it backs off and flags the delta
__device__ __forceinline__ bool claim_point(const PoolArgs &a, int p) {
    if ((unsigned)p >= (unsigned)a.pt_cap) {
        atomicOr(a.status, kStIndex);
        return false;
    }
    if (atomicExch(a.pt_stamp + p, a.stamp) == a.stamp) {
        atomicOr(a.status, kStTwice);
        return false;
    }
    return true;
}

// position of keyframe k in a list of c entries (c if absent; a keyframe occurs at most once): eight independent loads per
// step instead of a dependent chain of c, newest entries first (culling the newest keyframe's observations is O(1))
__device__ __forceinline__ int find_keyframe(const int *__restrict__ list, int c, int k) {
    for (int j = c; j > 0; j -= 8) {
        int v[8];
#pragma unroll
        for (int q = 0; q < 8; q++) v[q] = j - 1 - q >= 0 ? list[j - 1 - q] : ~k;
#pragma unroll
        for (int q = 0; q < 8; q++)
            if (v[q] == k) return j - 1 - q;
    }
    return c;
}

// MapPoint::EraseObservation(pKF), src/MapPoint.cc:111-141: the entry of keyframe kf leaves the list, the rest closes up
// one atomic per warp on the live-observation counter (800k requests on one address would serialise in L2)
__device__ __forceinline__ void live_add(int *ctr, int delta) {
    const unsigned m = __activemask();
    const int tot = __reduce_add_sync(m, delta);
    if ((threadIdx.x & 31) == (unsigned)(__ffs(m) - 1) && tot) atomicAdd(ctr, tot);
}

__global__ void __launch_bounds__(kThreads)
k_map_erase(PoolArgs a, const int *__restrict__ pt, const int *__restrict__ kf, int n) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int p = __ldg(pt + i), k = __ldg(kf + i);
    int gone = 0;
    if (claim_point(a, p)) {
        const int s = a.pt_start[p], c = a.pt_cnt[p];
        int j = find_keyframe(a.pool_kf + s, c, k);
        if (j < c) {  // (:116: nothing happens when the point has no observation in that keyframe)
            for (; j + 1 < c; j++) {
                a.pool_kf[s + j] = a.pool_kf[s + j + 1];
                a.pool_uv[s + j] = a.pool_uv[s + j + 1];
            }
            a.pt_cnt[p] = c - 1;
            gone = 1;
        }
    }
    live_add(a.ctr + kCtrLive, -gone);
}

// MapPoint::SetBadFlag, src/MapPoint.cc:151-168: mObservations.clear()
__global__ void __launch_bounds__(kThreads)
k_map_bad(PoolArgs a, const int *__restrict__ pt, int n) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int p = __ldg(pt + i);
    if ((unsigned)p >= (unsigned)a.pt_cap) {
        atomicOr(a.status, kStIndex);
        return;
    }
    const int c = atomicExch(a.pt_cnt + p, 0);
    if (c) atomicSub(a.ctr + kCtrLive, c);  // (a few points per step)
}

// MapPoint::AddObservation(pKF, idx), src/MapPoint.cc:98-109
__global__ void __launch_bounds__(kThreads)
k_map_add(PoolArgs a, const int *__restrict__ pt, const int *__restrict__ kf, const int *__restrict__ fid, int n) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int p = __ldg(pt + i), k = __ldg(kf + i), f = __ldg(fid + i);
    int added = 0;
    if ((unsigned)k >= (unsigned)a.n_kf || (unsigned)f >= (unsigned)a.kp_stride) {
        atomicOr(a.status, kStIndex);
    } else if (claim_point(a, p)) {
        int s = a.pt_start[p];
        const int c = a.pt_cnt[p], room = a.pt_room[p];
        bool ok = find_keyframe(a.pool_kf + s, c, k) == c;  // :101-102 no-op when the point is already observed in this keyframe
        if (ok && c == room) {  // the run is full: move the list to the tail, with twice the room
            const int nroom = room < kMinRoom ? kMinRoom : 2 * room;
            const int ns = atomicAdd(a.ctr + kCtrTail, nroom);
            if ((long long)ns + nroom > (long long)a.ctr[kCtrCap]) {
                atomicOr(a.status, kStPool);  // (the host keeps the pool ahead of demand; see map_prepare)
                ok = false;
            } else {
                for (int j = 0; j < c; j++) {
                    a.pool_kf[ns + j] = a.pool_kf[s + j];
                    a.pool_uv[ns + j] = a.pool_uv[s + j];
                }
                a.pt_start[p] = ns;
                a.pt_room[p] = nroom;
                s = ns;
            }
        }
        if (ok) {
            a.pool_kf[s + c] = k;
            a.pool_uv[s + c] = __ldg(a.kp_tab + (size_t)k * a.kp_stride + f);
            a.pt_cnt[p] = c + 1;
            added = 1;
        }
    }
    live_add(a.ctr + kCtrLive, added);
}

// bulk load: points [first, first + count) get fresh runs of (count + slack) entries at the tail, in point order
__global__ void k_map_bulk_base(int *ctr, int need, int *status) {
    const int base = atomicAdd(ctr + kCtrTail, need);
    ctr[kCtrBase] = base;
    if ((long long)base + need > (long long)ctr[kCtrCap]) atomicOr(status, kStPool);
}

__device__ __forceinline__ int bulk_room(int c, int slack_percent) {
    const int extra = (int)(((long long)c * slack_percent + 99) / 100);
    return c + (slack_percent > 0 && extra < 2 ? 2 : extra);
}

__global__ void __launch_bounds__(kThreads)
k_map_bulk_points(PoolArgs a, int first, int count, const int *__restrict__ obs_ptr, const int *__restrict__ run_ptr) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= count || (a.status[0] & kStPool)) return;
    const int c = __ldg(obs_ptr + i + 1) - __ldg(obs_ptr + i);
    const int old = a.pt_cnt[first + i];
    a.pt_start[first + i] = a.ctr[kCtrBase] + __ldg(run_ptr + i);
    a.pt_cnt[first + i] = c;
    a.pt_room[first + i] = __ldg(run_ptr + i + 1) - __ldg(run_ptr + i);
    if (c != old) atomicAdd(a.ctr + kCtrLive, c - old);
}

__global__ void __launch_bounds__(kThreads)
k_map_bulk_entries(PoolArgs a, int first, int count, const int *__restrict__ obs_ptr, const int2 *__restrict__ ref) {
    // one warp per point: lanes stride over the point's list
    const int w = (blockIdx.x * kThreads + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= count || (a.status[0] & kStPool)) return;
    const int e0 = __ldg(obs_ptr + w), e1 = __ldg(obs_ptr + w + 1);
    const int s = a.pt_start[first + w];
    for (int e = e0 + lane; e < e1; e += 32) {
        int2 r = __ldg(ref + e);
        if ((unsigned)r.x >= (unsigned)a.n_kf || (unsigned)r.y >= (unsigned)a.kp_stride) {
            atomicOr(a.status, kStIndex);
            r = make_int2(0, 0);
        }
        a.pool_kf[s + (e - e0)] = r.x;
        a.pool_uv[s + (e - e0)] = __ldg(a.kp_tab + (size_t)r.x * a.kp_stride + r.y);
    }
}

__global__ void k_map_set_word(int *dst, int v) { *dst = v; }
__global__ void k_map_set_header(MapHeader *dst, MapHeader h) { *dst = h; }

// export of observation lists (tests / snapshot files): counts, then entries
__global__ void __launch_bounds__(kThreads)
k_map_export_counts(const int *__restrict__ ids, int n, const int *__restrict__ pt_cnt, int pt_cap, int *__restrict__ out_cnt,
                    int *__restrict__ status) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int p = __ldg(ids + i);
    if ((unsigned)p >= (unsigned)pt_cap) {
        atomicOr(status, kStIndex);
        out_cnt[i] = 0;
        return;
    }
    out_cnt[i] = pt_cnt[p];
}

__global__ void __launch_bounds__(kThreads)
k_map_export_entries(const int *__restrict__ ids, int n, const int *__restrict__ pt_start, const int *__restrict__ pool_kf,
                     const float2 *__restrict__ pool_uv, const float *__restrict__ pt_xyz, int pt_cap,
                     const int *__restrict__ out_ptr, int *__restrict__ out_kf, float2 *__restrict__ out_uv,
                     float *__restrict__ out_xyz, long long cap) {
    const int w = (blockIdx.x * kThreads + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    const int p = __ldg(ids + w);
    if ((unsigned)p >= (unsigned)pt_cap) return;
    const int e0 = __ldg(out_ptr + w), e1 = __ldg(out_ptr + w + 1), s = pt_start[p];
    for (int e = e0 + lane; e < e1 && e < cap; e += 32) {
        out_kf[e] = pool_kf[s + (e - e0)];
        out_uv[e] = pool_uv[s + (e - e0)];
    }
    if (out_xyz && lane < 3) out_xyz[3 * (size_t)w + lane] = pt_xyz[3 * (size_t)p + lane];
}

// move a device array to a larger allocation, stream-ordered on ctx->stream (no host synchronisation)
template <typename T>
int grow_array(Ctx *ctx, T *&p, size_t old_n, size_t new_n, bool zero_tail) {
    T *q = nullptr;
    LCCRF_TRY(dev_alloc(ctx, (void **)&q, new_n * sizeof(T)));
    if (p && old_n) LCCRF_CUDA(cudaMemcpyAsync(q, p, old_n * sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream));
    if (zero_tail && new_n > old_n) LCCRF_CUDA(cudaMemsetAsync(q + old_n, 0, (new_n - old_n) * sizeof(T), ctx->stream));
    dev_free(ctx, p);
    p = q;
    return LCCRF_OK;
}

PoolArgs pool_args(DevMap *m) {
    PoolArgs a;
    a.pt_start = m->pt_start;
    a.pt_cnt = m->pt_cnt;
    a.pt_room = m->pt_room;
    a.pt_stamp = m->pt_stamp;
    a.pool_kf = m->pool_kf;
    a.pool_uv = (float2 *)m->pool_uv;
    a.ctr = m->d_ctr;
    a.status = m->ctx->d_status;
    a.kp_tab = (const float2 *)m->kp_tab;
    a.kp_stride = m->kp_stride;
    a.n_kf = m->n_kf;
    a.pt_cap = m->pt_cap;
    a.stamp = 0;
    return a;
}

int reserve_keyframes(DevMap *m, int n) {
    if (n <= m->kf_cap) return LCCRF_OK;
    Ctx *ctx = m->ctx;
    long long cap = m->kf_cap ? 2LL * m->kf_cap : 64;
    if (cap < n) cap = n;
    if (cap * (long long)m->kp_stride > (1LL << 33)) return fail(LCCRF_ERR_ARG, "keyframe keypoint table would exceed 2^33 keypoints");
    LCCRF_TRY(grow_array(ctx, m->kf_packed, (size_t)m->kf_cap, (size_t)cap, true));
    LCCRF_TRY(grow_array(ctx, m->kp_tab, (size_t)m->kf_cap * m->kp_stride * 2, (size_t)cap * m->kp_stride * 2, true));
    m->kf_cap = (int)cap;
    return map_publish(m);
}

// refresh the host's view of the device counters if the last snapshot has landed; request a new one
int poll_counters(DevMap *m, bool request) {
    if (m->ctr_pending && cudaEventQuery(m->ctr_ev) == cudaSuccess) {
        m->tail_seen = m->h_ctr[kCtrTail];
        m->ctr_pending = false;
    }
    if (request && !m->ctr_pending) {
        LCCRF_CUDA(cudaMemcpyAsync(m->h_ctr, m->d_ctr, 4 * sizeof(int), cudaMemcpyDeviceToHost, m->ctx->stream));
        LCCRF_CUDA(cudaEventRecord(m->ctr_ev, m->ctx->stream));
        m->ctr_pending = true;
    }
    return LCCRF_OK;
}

}  // namespace

int map_create(Ctx *ctx, int kp_stride, DevMap **out) {
    auto *m = new DevMap();
    m->ctx = ctx;
    m->kp_stride = kp_stride;
    int rc = dev_alloc(ctx, (void **)&m->d_hdr, sizeof(MapHeader), true);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&m->d_ctr, 4 * sizeof(int), true);
    if (rc == LCCRF_OK && (cudaHostAlloc((void **)&m->h_ctr, 4 * sizeof(int), cudaHostAllocDefault) != cudaSuccess ||
                           cudaEventCreateWithFlags(&m->ctr_ev, cudaEventDisableTiming) != cudaSuccess ||
                           cudaStreamCreateWithFlags(&m->mstream, cudaStreamNonBlocking) != cudaSuccess ||
                           cudaEventCreateWithFlags(&m->ev_touch, cudaEventDisableTiming) != cudaSuccess ||
                           cudaEventCreateWithFlags(&m->ev_mut, cudaEventDisableTiming) != cudaSuccess))
        rc = fail(LCCRF_ERR_CUDA, "map: pinned counters / event allocation failed");
    if (rc != LCCRF_OK) {
        map_destroy(m);
        return rc;
    }
    memset(m->h_ctr, 0, 4 * sizeof(int));
    *out = m;
    return LCCRF_OK;
}

void map_destroy(DevMap *m) {
    if (!m) return;
    Ctx *ctx = m->ctx;
    cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (m->mstream) cudaStreamSynchronize(m->mstream);
    dev_free(ctx, m->kf_packed);
    dev_free(ctx, m->kp_tab);
    dev_free(ctx, m->d_hdr);
    dev_free(ctx, m->pt_xyz);
    dev_free(ctx, m->pt_start);
    dev_free(ctx, m->pt_cnt);
    dev_free(ctx, m->pt_room);
    dev_free(ctx, m->pt_stamp);
    dev_free(ctx, m->pool_kf);
    dev_free(ctx, m->pool_uv);
    dev_free(ctx, m->d_ctr);
    if (m->h_ctr) cudaFreeHost(m->h_ctr);
    if (m->ctr_ev) cudaEventDestroy(m->ctr_ev);
    if (m->ev_touch) cudaEventDestroy(m->ev_touch);
    if (m->ev_mut) cudaEventDestroy(m->ev_mut);
    cudaStreamSynchronize(ctx->stream);  // the stream-ordered frees above
    if (m->mstream) cudaStreamDestroy(m->mstream);
    delete m;
}

int map_begin_main_access(DevMap *m) {
    LCCRF_CUDA(cudaStreamWaitEvent(m->ctx->stream, m->ev_mut, 0));
    return LCCRF_OK;
}

int map_end_main_access(DevMap *m) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    LCCRF_CUDA(cudaStreamIsCapturing(m->ctx->stream, &cs));
    if (cs == cudaStreamCaptureStatusActive)  // every replay of the graph records the event behind the unary kernel
        LCCRF_CUDA(cudaEventRecordWithFlags(m->ev_touch, m->ctx->stream, cudaEventRecordExternal));
    else
        LCCRF_CUDA(cudaEventRecord(m->ev_touch, m->ctx->stream));
    return LCCRF_OK;
}

int map_begin_async_mut(DevMap *m) {
    LCCRF_CUDA(cudaStreamWaitEvent(m->mstream, m->ev_touch, 0));
    return LCCRF_OK;
}

int map_end_async_mut(DevMap *m) {
    LCCRF_CUDA(cudaEventRecord(m->ev_mut, m->mstream));
    return LCCRF_OK;
}

int map_publish(DevMap *m) {
    Ctx *ctx = m->ctx;
    MapHeader h;
    h.kf_packed = m->kf_packed;
    h.pt_xyz = m->pt_xyz;
    h.pt_start = m->pt_start;
    h.pt_cnt = m->pt_cnt;
    h.pool_kf = m->pool_kf;
    h.pool_uv = m->pool_uv;
    h.n_kf = m->n_kf;
    { LCCRF_KERNEL(ctx, "k_map_set_header"); k_map_set_header<<<1, 1, 0, ctx->stream>>>(m->d_hdr, h); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int map_reserve_points(DevMap *m, int n) {
    if (n <= m->pt_cap) return LCCRF_OK;
    Ctx *ctx = m->ctx;
    long long cap = m->pt_cap ? 2LL * m->pt_cap : 4096;
    if (cap < n) cap = n;
    if (cap > (1LL << 30)) return fail(LCCRF_ERR_ARG, "more than 2^30 map points");
    LCCRF_TRY(grow_array(ctx, m->pt_xyz, (size_t)m->pt_cap * 3, (size_t)cap * 3, true));
    LCCRF_TRY(grow_array(ctx, m->pt_start, (size_t)m->pt_cap, (size_t)cap, true));
    LCCRF_TRY(grow_array(ctx, m->pt_cnt, (size_t)m->pt_cap, (size_t)cap, true));
    LCCRF_TRY(grow_array(ctx, m->pt_room, (size_t)m->pt_cap, (size_t)cap, true));
    LCCRF_TRY(grow_array(ctx, m->pt_stamp, (size_t)m->pt_cap, (size_t)cap, true));
    m->pt_cap = (int)cap;
    return map_publish(m);
}

// make the pool hold at least `entries` entries (stream-ordered move)
int map_reserve_pool(DevMap *m, long long entries) {
    if (entries <= m->pool_cap) return LCCRF_OK;
    Ctx *ctx = m->ctx;
    long long cap = m->pool_cap ? 2 * m->pool_cap : (1 << 16);
    if (cap < entries) cap = entries;
    if (cap > 0x7fffffffLL) cap = 0x7fffffffLL;
    if (cap < entries) return fail(LCCRF_ERR_ARG, "observation pool would exceed 2^31 entries");
    LCCRF_TRY(grow_array(ctx, m->pool_kf, (size_t)m->pool_cap, (size_t)cap, false));
    LCCRF_TRY(grow_array(ctx, m->pool_uv, (size_t)m->pool_cap * 2, (size_t)cap * 2, false));
    m->pool_cap = cap;
    { LCCRF_KERNEL(ctx, "k_map_set_word"); k_map_set_word<<<1, 1, 0, ctx->stream>>>(m->d_ctr + kCtrCap, (int)cap); }
    LCCRF_CUDA(cudaGetLastError());
    return map_publish(m);
}

int map_prepare(DevMap *m, const lccrf_map_delta &h) {
    if (h.kf_count < 0 || h.kf_first < 0 || h.n_pose < 0 || h.n_xyz < 0 || h.n_erase < 0 || h.n_bad < 0 || h.n_add < 0)
        return fail(LCCRF_ERR_ARG, "map delta: negative count");
    if (h.kf_count > 0) {
        if (!h.kf_pose || !h.kf_intr || !h.kf_bounds) return fail(LCCRF_ERR_ARG, "map delta: new keyframes need pose, intrinsics and bounds");
        if ((long long)h.kf_first + h.kf_count > 0x7fffffffLL) return fail(LCCRF_ERR_ARG, "map delta: keyframe id overflow");
        LCCRF_TRY(reserve_keyframes(m, h.kf_first + h.kf_count));
        // one camera for every keyframe (a monocular / RGB-D sequence): intrinsics and bounds travel as kernel parameters
        for (int k = 0; k < h.kf_count; k++) {
            float c8[8];
            memcpy(c8, h.kf_intr + 4 * (size_t)k, 16);
            memcpy(c8 + 4, h.kf_bounds + 4 * (size_t)k, 16);
            if (!m->cam_set) {
                memcpy(m->cam8, c8, sizeof(c8));
                m->cam_set = true;
            } else if (m->ucam && memcmp(m->cam8, c8, sizeof(c8)) != 0) {
                m->ucam = false;
            }
        }
        if (h.kf_first + h.kf_count > m->n_kf) m->n_kf = h.kf_first + h.kf_count;
    }
    if (h.n_pose > 0 && !h.pose) return fail(LCCRF_ERR_ARG, "map delta: pose is NULL");
    if (h.n_xyz > 0) {
        if (!h.xyz) return fail(LCCRF_ERR_ARG, "map delta: xyz is NULL");
        if (!h.xyz_id) {
            LCCRF_TRY(map_reserve_points(m, h.n_xyz));
            if (h.n_xyz > m->n_pt) m->n_pt = h.n_xyz;
        }
        // explicit ids: the caller creates points densely; ids beyond the capacity are flagged on the device unless
        // the capacity was raised first (lccrf_map_set_observations / an id-less xyz block / the first delta below)
    }
    if (h.n_erase > 0 && (!h.erase_pt || !h.erase_kf)) return fail(LCCRF_ERR_ARG, "map delta: erase arrays are NULL");
    for (int which = 0; which < 2; which++) {
        const int ns = which ? h.n_add_seg : h.n_erase_seg, total = which ? h.n_add : h.n_erase;
        const int *sp = which ? h.add_seg_ptr : h.erase_seg_ptr;
        if (ns < 0 || (ns > 0 && !sp)) return fail(LCCRF_ERR_ARG, "map delta: segment pointer array is NULL");
        if (ns > 0) {
            if (sp[0] != 0 || sp[ns] != total) return fail(LCCRF_ERR_ARG, "map delta: segments must span the whole list");
            for (int g = 0; g < ns; g++)
                if (sp[g + 1] < sp[g]) return fail(LCCRF_ERR_ARG, "map delta: segment boundaries must be non-decreasing");
        }
    }
    if (h.n_bad > 0 && !h.bad_pt) return fail(LCCRF_ERR_ARG, "map delta: bad_pt is NULL");
    if (h.n_add > 0) {
        if (!h.add_pt || !h.add_kf || !h.add_fid) return fail(LCCRF_ERR_ARG, "map delta: add arrays are NULL");
        // Pool head-room.  A single append moves at most one list (twice its room).  The host sees the tail with a lag
        // of a few steps (asynchronous snapshots), so it keeps the pool at least half empty beyond that view plus this
        // delta's minimum need; a list that outgrows even that is reported (status bit 16), never written out of bounds.
        poll_counters(m, false);
        const long long known = m->tail_seen + m->tail_unseen;
        const long long want = 2 * known + 8LL * h.n_add + (1 << 16);
        if (want > m->pool_cap) LCCRF_TRY(map_reserve_pool(m, want));
    }
    return LCCRF_OK;
}

size_t delta_stage_bytes(const lccrf_map_delta &d, int kp_stride, bool with_keypoints) {
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    size_t n = 0;
    n += al((size_t)d.kf_count * 48) + al((size_t)d.kf_count * 16) * 2;
    if (with_keypoints && d.kf_keypoints) n += al((size_t)d.kf_count * kp_stride * 8);
    n += al((size_t)d.n_pose * 4) + al((size_t)d.n_pose * 48);
    n += al((size_t)d.n_xyz * 4) + al((size_t)d.n_xyz * 12);
    n += al((size_t)d.n_erase * 4) * 2 + al((size_t)d.n_bad * 4) + al((size_t)d.n_add * 4) * 3;
    return n + 256;
}

int delta_stage(const lccrf_map_delta &d, int kp_stride, bool with_keypoints, char *base, cudaStream_t st, DeltaDev *out) {
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

int delta_grow_points(DevMap *m, const lccrf_map_delta &d) {
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

int map_apply_dev(DevMap *m, const DeltaDev &d, const float *kp_host) {
    Ctx *ctx = m->ctx;
    cudaStream_t st = ctx->stream;
    if (d.kf_count > 0) {
        { LCCRF_KERNEL(ctx, "k_map_set_kf");
          k_map_set_kf<<<cdiv(d.kf_count, kThreads), kThreads, 0, st>>>(m->kf_packed, d.kf_pose, d.kf_intr, d.kf_bounds, d.kf_first, d.kf_count); }
        const size_t row = (size_t)m->kp_stride * 2 * sizeof(float);
        if (kp_host)
            LCCRF_CUDA(cudaMemcpyAsync(m->kp_tab + (size_t)d.kf_first * m->kp_stride * 2, kp_host, row * d.kf_count, cudaMemcpyHostToDevice, st));
        else if (d.kf_keypoints)
            LCCRF_CUDA(cudaMemcpyAsync(m->kp_tab + (size_t)d.kf_first * m->kp_stride * 2, d.kf_keypoints, row * d.kf_count, cudaMemcpyDeviceToDevice, st));
        LCCRF_TRY(map_publish(m));  // the keyframe count
    }
    if (d.n_pose > 0) {
        LCCRF_KERNEL(ctx, "k_map_set_pose");
        k_map_set_pose<<<cdiv(d.n_pose, kThreads), kThreads, 0, st>>>(m->kf_packed, d.pose_kf, d.pose, d.n_pose, m->n_kf, ctx->d_status);
    }
    if (d.n_xyz > 0) {
        LCCRF_KERNEL(ctx, "k_map_set_xyz");
        k_map_set_xyz<<<cdiv(d.n_xyz, kThreads), kThreads, 0, st>>>(m->pt_xyz, d.xyz_id, d.xyz, d.n_xyz, m->pt_cap, ctx->d_status);
    }
    PoolArgs a = pool_args(m);
    for (size_t g = 0; d.n_erase > 0 && g < (d.erase_seg.empty() ? 1 : d.erase_seg.size() - 1); g++) {
        const int e0 = d.erase_seg.empty() ? 0 : d.erase_seg[g], e1 = d.erase_seg.empty() ? d.n_erase : d.erase_seg[g + 1];
        if (e1 <= e0) continue;
        a.stamp = ++m->epoch;
        LCCRF_KERNEL(ctx, "k_map_erase");
        k_map_erase<<<cdiv(e1 - e0, kThreads), kThreads, 0, st>>>(a, d.erase_pt + e0, d.erase_kf + e0, e1 - e0);
    }
    if (d.n_bad > 0) {
        LCCRF_KERNEL(ctx, "k_map_bad");
        k_map_bad<<<cdiv(d.n_bad, kThreads), kThreads, 0, st>>>(a, d.bad_pt, d.n_bad);
    }
    for (size_t g = 0; d.n_add > 0 && g < (d.add_seg.empty() ? 1 : d.add_seg.size() - 1); g++) {
        const int e0 = d.add_seg.empty() ? 0 : d.add_seg[g], e1 = d.add_seg.empty() ? d.n_add : d.add_seg[g + 1];
        if (e1 <= e0) continue;
        a.stamp = ++m->epoch;
        LCCRF_KERNEL(ctx, "k_map_add");
        k_map_add<<<cdiv(e1 - e0, kThreads), kThreads, 0, st>>>(a, d.add_pt + e0, d.add_kf + e0, d.add_fid + e0, e1 - e0);
    }
    if (d.n_add > 0) LCCRF_TRY(poll_counters(m, true));
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

// obs_ptr_dev [count+1], obs_ref_dev [nnz][2] on the device; run_ptr (exclusive prefix of the runs' rooms) is built on
// the host by the caller and passed in obs_ptr_dev + count + 1 .. (see lccrf_map_set_observations)
int map_bulk_observations(DevMap *m, int pt_first, int count, const int *obs_ptr_dev, const int *obs_ref_dev, long long nnz,
                          int slack_percent) {
    (void)slack_percent;
    (void)nnz;
    Ctx *ctx = m->ctx;
    cudaStream_t st = ctx->stream;
    PoolArgs a = pool_args(m);
    const int *run_ptr = obs_ptr_dev + count + 1;
    { LCCRF_KERNEL(ctx, "k_map_bulk_points");
      k_map_bulk_points<<<cdiv(count, kThreads), kThreads, 0, st>>>(a, pt_first, count, obs_ptr_dev, run_ptr); }
    { LCCRF_KERNEL(ctx, "k_map_bulk_entries");
      k_map_bulk_entries<<<cdiv((long long)count * 32, kThreads), kThreads, 0, st>>>(a, pt_first, count, obs_ptr_dev, (const int2 *)obs_ref_dev); }
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

// (used by lccrf_map_set_observations) reserve `need` entries at the tail; the base lands in d_ctr[kCtrBase]
int map_bulk_reserve(DevMap *m, long long need) {
    Ctx *ctx = m->ctx;
    poll_counters(m, false);
    const long long known = m->tail_seen + m->tail_unseen;
    if (known + need + (1 << 16) > m->pool_cap) LCCRF_TRY(map_reserve_pool(m, 2 * (known + need) + (1 << 16)));
    if (need > 0x7fffffffLL) return fail(LCCRF_ERR_ARG, "bulk load exceeds 2^31 observations");
    { LCCRF_KERNEL(ctx, "k_map_bulk_base"); k_map_bulk_base<<<1, 1, 0, ctx->stream>>>(m->d_ctr, (int)need, ctx->d_status); }
    m->tail_unseen += need;
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int map_export_dev(DevMap *m, int n, const int *ids_dev, int *cnt_dev) {
    Ctx *ctx = m->ctx;
    LCCRF_TRY(map_begin_main_access(m));
    LCCRF_KERNEL(ctx, "k_map_export_counts");
    k_map_export_counts<<<cdiv(n, kThreads), kThreads, 0, ctx->stream>>>(ids_dev, n, m->pt_cnt, m->pt_cap, cnt_dev, ctx->d_status);
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int map_export_entries_dev(DevMap *m, int n, const int *ids_dev, const int *ptr_dev, int *kf_dev, float *uv_dev, float *xyz_dev,
                           long long cap) {
    Ctx *ctx = m->ctx;
    LCCRF_KERNEL(ctx, "k_map_export_entries");
    k_map_export_entries<<<cdiv((long long)n * 32, kThreads), kThreads, 0, ctx->stream>>>(
        ids_dev, n, m->pt_start, m->pool_kf, (const float2 *)m->pool_uv, m->pt_xyz, m->pt_cap, ptr_dev, kf_dev, (float2 *)uv_dev,
        xyz_dev, cap);
    LCCRF_CUDA(cudaGetLastError());
    return LCCRF_OK;
}

int map_counters(DevMap *m, long long *tail, long long *live) {  // synchronises
    Ctx *ctx = m->ctx;
    LCCRF_CUDA(cudaStreamSynchronize(m->mstream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    int h[4];
    LCCRF_CUDA(cudaMemcpy(h, m->d_ctr, sizeof(h), cudaMemcpyDeviceToHost));
    m->tail_seen = h[kCtrTail];
    m->tail_unseen = 0;
    m->ctr_pending = false;
    if (tail) *tail = h[kCtrTail];
    if (live) *live = h[kCtrLive];
    return LCCRF_OK;
}

}  // namespace lccrf
