/*
 * lccrf.h -- C ABI of liblccrf.so: the B200 (sm_100a) implementation of LC-CRF-SLAM's
 * data-parallel hot path (fully connected CRF over permutohedral lattices + long-term unary).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  Every entry
 * point names the reference interface it replaces (paths relative to the LC-CRF-SLAM tree).
 * The C++ header mirror in lc-crf-slam_b200/densecrf/ (DenseCRF3D<M>, PottsPotential3D<M,F>,
 * DenseCRFCPU<M>, PottsPotentialCPU<M,F>, PermutohedralLatticeCPU) forwards to these calls,
 * so src/Tracking.cc:1919-1930 and Thirdparty/DenseCRF/examples/example_cpu.cpp:80-102
 * compile unchanged.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - All pointers are HOST pointers unless the name says "_dev".
 *   - Return value: 0 = LCCRF_OK, negative = error; lccrf_last_error() gives the message
 *     (thread-local).  The reference API is all-void with no validation (SURVEY 8b "Errors");
 *     the C++ mirror aborts with the message on a non-zero status.
 *   - There is NO CPU fallback: every computing call fails with LCCRF_ERR_CUDA when no
 *     sm_100 device / driver is usable.
 *   - N == 0 is a valid no-op everywhere.
 *   - Thread safety: one lccrf_ctx per host thread (or external locking); handles created
 *     from a ctx share its stream.
 */
#ifndef LCCRF_H
#define LCCRF_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCCRF_OK 0
#define LCCRF_ERR_ARG (-1)     /* bad argument (null pointer, unsupported d / L, ...) */
#define LCCRF_ERR_CUDA (-2)    /* CUDA runtime / driver failure, or no device */
#define LCCRF_ERR_STATE (-3)   /* call sequence error (e.g. step before start) */
#define LCCRF_ERR_RANGE (-4)   /* a lattice key left the reference's `short` range (permutohedral_cpu.h:373) */

#define LCCRF_MAX_D 7          /* feature dimensions supported by the lattice (reference uses 2 and 5) */
#define LCCRF_MAX_L 64         /* labels (reference uses 2; the golden demo uses 21) */
#define LCCRF_MAX_K 8          /* pairwise potentials per CRF */

typedef struct lccrf_ctx lccrf_ctx;
typedef struct lccrf_lattice lccrf_lattice;
typedef struct lccrf_crf lccrf_crf;
typedef struct lccrf_frames lccrf_frames;

/* ---------------------------------------------------------------- context ---------------- */
const char *lccrf_version(void);
const char *lccrf_last_error(void);
int lccrf_device_count(void);
/* one context per GPU (and per host thread): owns a stream, memory pools, workspaces */
int lccrf_ctx_create(int device, lccrf_ctx **out);
void lccrf_ctx_destroy(lccrf_ctx *ctx);
/* run on an externally owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); NULL = own stream */
int lccrf_ctx_set_stream(lccrf_ctx *ctx, void *cuda_stream);
int lccrf_ctx_sync(lccrf_ctx *ctx);
/* number of liblccrf kernels launched on this context so far (bench.py "gpu_launches") */
uint64_t lccrf_ctx_kernel_launches(const lccrf_ctx *ctx);
/* diagnostic: synchronises and counts the slots of the context's lattice-build hash scratch that are not empty.  Every
 * build empties the slots it used, so the count is 0 whenever no build is in flight. */
int lccrf_ctx_build_scratch_in_use(lccrf_ctx *ctx, long long *slots);
/* option knobs (default):
 *   "ordered_splat" (1)  1: every lattice vertex sums its contributions in point order -- marginals bit-identical to the
 *                        reference; 0: fixed-shape tree reduction, 3x faster splat, marginals within 1e-4 of the reference
 *                        at frame-sized problems but not at N = 100k x 64 (DESIGN.md 3.2)
 *   "graphs" (1)         CUDA-graph replay of lccrf_frames_run / submit once a launch sequence repeats its shape
 *   "concurrent" (1)     the two pairwise kernels of a frame batch on two graph branches
 *   "split_splat" (1)    with "concurrent": a lattice's short-row splat runs beside its long-row scan kernels
 *   "fused" (1)          fused point pass (slice of all lattices + Potts apply + softmax) for two labels
 *   "bulk_blur" (1)      element-parallel blur streams its operands with cp.async.bulk (0: plain vector loads)
 *   "map_slack" (0)      spare room, in percent, behind every list of lccrf_map_set_observations
 *   "profile" (0)        per-kernel CUDA-event timing, see lccrf_ctx_profile_report
 *   "trace" (0)          host-side phase times of the pipelined submissions on stderr */
int lccrf_ctx_set_option(lccrf_ctx *ctx, const char *name, int value);
/* Per-kernel timing.  With option "profile" = 1 every kernel launch is bracketed by two CUDA events on
 * the launching stream (graphs are bypassed while profiling).  The report synchronises, writes one line
 * per kernel name -- "name launches total_ms" -- into buf (NUL-terminated, truncated to cap) and
 * clears the records.  Returns the number of distinct kernels, negative on error. */
int lccrf_ctx_profile_report(lccrf_ctx *ctx, char *buf, int cap);

/* ---------------------------------------------------------------- lattice ---------------- */
/* Replaces PermutohedralLatticeCPU::init(feature, feature_size, N)
 *   Thirdparty/DenseCRF/include/permutohedral_cpu.h:241-424 (SSE branch, incl. the phantom
 *   lanes k in [N, ceil4(N)) that the reference inserts into its hash table, :294-299,364-377).
 * features: [N*d] row-major.  Vertex ids, barycentric bit patterns and the neighbour table are
 * bit-identical to the reference. */
int lccrf_lattice_create(lccrf_ctx *ctx, const float *features, int d, int N, lccrf_lattice **out);
void lccrf_lattice_destroy(lccrf_lattice *lat);
/* N_, d_, M_ of permutohedral_cpu.h:187 */
int lccrf_lattice_sizes(const lccrf_lattice *lat, int *N, int *d, int *V);
/* offset_[N*(d+1)], barycentric_[N*(d+1)] (permutohedral_cpu.h:375-376) and
 * blur_neighbors_[(d+1)*V] as {n1,n2} int pairs indexed [j*V+i] (:418-419).  Any pointer may be NULL. */
int lccrf_lattice_export(const lccrf_lattice *lat, int *offset, float *bary, int *nbr);
/* Replaces PermutohedralLatticeCPU::compute(out, in, value_size) with default windowing
 *   permutohedral_cpu.h:634-699.  in/out: [N*L]; out may alias in (pairwise3d.h:24). */
int lccrf_lattice_filter(lccrf_lattice *lat, float *out, const float *in, int L);
/* ... with its windowing arguments (permutohedral_cpu.h:634-637): only points [in_offset, in_offset + in_size) are
 * splatted (in: [in_size*L]) and only points [out_offset, out_offset + out_size) are sliced (out: [out_size*L]);
 * -1 = up to the last point.  Bit-identical to the reference: a window is a zero-padded input (a running sum that
 * starts at +0 is unchanged by +-0 addends) and a cropped output. */
int lccrf_lattice_filter_window(lccrf_lattice *lat, float *out, const float *in, int L, int in_offset, int out_offset,
                                int in_size, int out_size);
/* diagnostics of the ordered splat's long rows, the counters of lccrf_frames_debug_counters: out8 = {#long rows,
 * #chunks, #pieces, compose tickets, chunk records applied in O(1), crossing windows applied, chunks summed for real,
 * zero chunks} (the last four accumulate over the filter calls since the lattice was built) */
int lccrf_lattice_debug_counters(const lccrf_lattice *lat, int *out8);

/* ---------------------------------------------------------------- dense CRF -------------- */
/* Replaces DenseCRF3D<M>(N) / DenseCRFCPU<M>(N)   densecrf3d.h:23-28, densecrf_cpu.h:22-27 */
int lccrf_crf_create(lccrf_ctx *ctx, int N, int L, lccrf_crf **out);
/* ~DenseCRF: also destroys the potentials it owns (densecrf_base.h:41-45) */
void lccrf_crf_destroy(lccrf_crf *crf);
/* setUnaryEnergy(const float*)   densecrf3d.h:41-43 ; unary: [N*L] */
int lccrf_crf_set_unary(lccrf_crf *crf, const float *unary);
/* setUnaryEnergyFromLabel(label, confidences)   densecrf3d.h:108-130.
 * The three energy tables are the values the reference computes at :109-114
 * (u = -log(1/M), n[m] = -log((1-c[m])/(M-1)), p[m] = -log(c[m])); the C++ mirror evaluates
 * them with the same expressions in the caller's translation unit.  label: [N], -1 = unknown. */
int lccrf_crf_set_unary_from_label(lccrf_crf *crf, const short *label, float u_energy,
                                   const float *n_energies, const float *p_energies);
/* SetUnaryEnergtForPositiveNode(idx, m, value)   densecrf3d.h:132-134 */
int lccrf_crf_set_unary_entry(lccrf_crf *crf, int idx, int m, float value);
/* addPairwiseEnergy(new PottsPotential3D<M,d>(features, N, w)) -- lattice build + norm_
 *   pairwise3d.h:20-28 (== pairwise_cpu.h:15-23) + densecrf_base.h:54.  features: [N*d]. */
int lccrf_crf_add_potts(lccrf_crf *crf, const float *features, int d, float w);
/* addPairwiseEnergy(PottsPotentialCPU<M,F>::FromImage<T>(W,H,weight,posdev,features,featuredev))
 *   pairwise_cpu.h:34-50; features assembled on the device.  img: [W*H*(F-2)] u8 or f32 (NULL if F==2). */
int lccrf_crf_add_potts_image(lccrf_crf *crf, int W, int H, float w, float posdev, const void *img,
                              int img_is_u8, int F, float featuredev);
/* startInference / stepInference(relax) / inference(n, with_map, relax)   densecrf_base.h:65-91 */
int lccrf_crf_start(lccrf_crf *crf);
int lccrf_crf_step(lccrf_crf *crf, float relax);
int lccrf_crf_inference(lccrf_crf *crf, int n_iterations, int with_map, float relax);
/* buildMap()   densecrf3d.h:137-151 (for the step-by-step API) */
int lccrf_crf_build_map(lccrf_crf *crf);
/* getMap() / getProbability(): library-owned HOST arrays, valid until the next call that
 * changes them or destroy (densecrf_base.h:74-75).  NULL before they exist. */
const short *lccrf_crf_map(lccrf_crf *crf);
const float *lccrf_crf_prob(lccrf_crf *crf);
/* lattice sizes of potential k (tests / diagnostics); number of potentials added so far */
int lccrf_crf_potts_vertices(const lccrf_crf *crf, int k, int *V);
int lccrf_crf_num_potts(const lccrf_crf *crf);

/* Plugin support: user-defined PairwisePotential::apply(out, in, tmp) on host pointers
 * (densecrf_base.h:12-19).  These expose the driver's pieces on host arrays so that the C++
 * mirror can interleave foreign potentials with built-in ones; all arithmetic still runs on
 * the GPU.
 *   potts_apply: PottsPotential3D::apply   pairwise3d.h:73-78   out[N*L] += w*norm*filter(in)
 *   exp_and_normalize: DenseCRF3D<M>::expAndNormalize   densecrf3d.h:71-98 */
int lccrf_crf_potts_apply(lccrf_crf *crf, int k, float *out, const float *in, float *tmp);
/*   step_init: DenseCRF3D<M>::stepInit   densecrf3d.h:155-158   next[N*L] = -unary
 *   set_prob:  overwrite current_ (the marginals) with host values after a host-driven step */
int lccrf_crf_step_init(lccrf_crf *crf, float *next);
int lccrf_crf_set_prob(lccrf_crf *crf, const float *prob);
int lccrf_exp_and_normalize(lccrf_ctx *ctx, float *out, const float *in, int N, int L, float scale,
                            float relax);

/* ---------------------------------------------------------------- long-term unary -------- */
/* TUM3.yaml:81-101 / Tracking.cc:151-171 */
typedef struct lccrf_slam_params {
    float w1, w2;
    float u_alpha, stdev_alpha; /* mRpjErrorMean, mRpjErrorStdev */
    float u_beta, stdev_beta;   /* mObservMean, mObservStdev */
    float u_gamma, stdev_gamma; /* mGcMean, mGcStdev (epipolar prior; not used on this path) */
    float point3d_stdev, point2d_stdev;
    float u_depth, pth, confidence;
    int iters;                  /* Tracking.cc:1929 */
} lccrf_slam_params;

/* Replaces Tracking::ComputeMapPointErrAndObserv over all N map points
 *   src/Tracking.cc:1803-1839, on a flat snapshot of the pointer graph (SURVEY 8a U1):
 *   xyz [N*3]; CSR obs_ptr [N+1]; obs_kf [nnz]; obs_uv [nnz*2]; kf_pose [nKF*12] rows of [Rcw|tcw];
 *   kf_intr [nKF*4] fx fy cx cy; kf_bounds [nKF*4] mnMinX mnMaxX mnMinY mnMaxY.
 * Out: observs [N] (as float, Tracking.cc:1867), error [N], depth [N].  Observations are
 * accumulated in CSR order (the reference iterates a std::map in pointer order). */
int lccrf_map_point_unary(lccrf_ctx *ctx, int N, const float *xyz, const int *obs_ptr, const int *obs_kf,
                          const float *obs_uv, int nKF, const float *kf_pose, const float *kf_intr,
                          const float *kf_bounds, float *observs, float *error, float *depth);
/* Replaces Tracking::RroughClassify   src/Tracking.cc:1961-2013.  p4: per-point epipolar
 * likelihood (double, mvFeatureMatchProb[fid]) or NULL when the map is empty (:1994). */
int lccrf_rough_classify(lccrf_ctx *ctx, int N, const float *observs, const float *error, const float *depth,
                         const double *p4, const lccrf_slam_params *prm, short *label);

/* ---------------------------------------------------------------- frontend (SURVEY 8f) --- */
/* Replaces Tracking::GetFeature2EpipolarDis   src/Tracking.cc:2030-2047, i.e. per match
 *   FundamentalMatrixEstimator::symmetricEpipolarDistance
 *     Thirdparty/graph-cut-ransac-master/include/fundamental_estimator.h:90-127   (double, incl. its y1-for-y2 quirk at :121)
 *   prob = exp(-(dis-mGcMean)^2 / (2*mGcStdev*mGcStdev))   Tracking.cc:2043.
 * M matches of `asso`: fid1 [M] feature id in the current frame (may be NULL when only the per-match outputs
 * are wanted), pt1 [M*2] = mCurrentFrame.mvKeysUn[fid1].pt, pt2 [M*2] = mLastFrame.mvKeysUn[fid2].pt,
 * F9 = fundModel.descriptor row-major.  Outputs (any may be NULL): dis/prob [M] per match, and dis_by_fid /
 * prob_by_fid [nFeat], the flat form of mvFeatureMatchDis / mvFeatureMatchProb -- features without a match
 * read 0.0, the value std::map::operator[] inserts at Tracking.cc:2003.  p4[i] = prob_by_fid[fid of point i]
 * is what lccrf_rough_classify takes. */
int lccrf_epipolar_prior(lccrf_ctx *ctx, int M, const int *fid1, const float *pt1, const float *pt2,
                         const double *F9, float u_gamma, float stdev_gamma, int nFeat, double *dis_by_fid,
                         double *prob_by_fid, double *dis, double *prob);
/* Replaces Tracking::BfMatch   src/Tracking.cc:1747-1766:
 *   cv::BFMatcher(cv::NORM_HAMMING).knnMatch(fl.mDescriptors, fr.mDescriptors, matches, 2) and the ratio test
 *   match[0].distance < match[1].distance * 0.6 (:1755, evaluated in double).
 * desc_q [nq*32], desc_t [nt*32]: 256-bit ORB descriptors (rows of the CV_8U x 32 cv::Mat).
 * match [nq]: asso[q] = train index of the accepted correspondence, -1 = rejected (or nt < 2).
 * knn (optional) [nq*4]: {d0, i0, d1, i1}, the two nearest train rows; equal distances keep the lower index
 * first (OpenCV's K-best insertion; pinned against cv2 in tests/golden).  n_match (optional): accepted count. */
int lccrf_bf_match(lccrf_ctx *ctx, int nq, const uint8_t *desc_q, int nt, const uint8_t *desc_t, double ratio,
                   int *match, int *knn, int *n_match);
/* B frame pairs in one launch (sequence replay: frame i against frame i-15, Tracking.cc:266-272): pair b owns
 * query rows [q_ptr[b], q_ptr[b+1]) and train rows [t_ptr[b], t_ptr[b+1]); indices in match / knn are local
 * to the pair's train range. */
int lccrf_bf_match_batch(lccrf_ctx *ctx, int B, const int *q_ptr, const uint8_t *desc_q, const int *t_ptr,
                         const uint8_t *desc_t, double ratio, int *match, int *knn, int *n_match);

/* ---------------------------------------------------------------- batched frames --------- */
/* B independent per-frame CRF problems (the body of Tracking::DynamicDetectionWithCRF,
 * src/Tracking.cc:1871-1930, for B frames at once): RroughClassify -> setUnaryEnergyFromLabel ->
 * appearanceKernel + smoothKernel -> inference(iters, true).  Points are concatenated; problem b
 * owns points [prob_ptr[b], prob_ptr[b+1]).  energies = {u, n, p} as in set_unary_from_label
 * with one shared confidence (Tracking.cc:1921). */
int lccrf_frames_create(lccrf_ctx *ctx, int B, const int *prob_ptr, const lccrf_slam_params *prm,
                        const float *energies3, lccrf_frames **out);
void lccrf_frames_destroy(lccrf_frames *fr);
/* per-frame vectors gathered at Tracking.cc:1849-1870: observs/error/depth [NT], kp2d [NT*2] */
int lccrf_frames_set_inputs(lccrf_frames *fr, const float *observs, const float *error, const float *depth,
                            const float *kp2d);
/* alternatively derive observs/error/depth on the device from a map snapshot (lccrf_map_point_unary layout);
 * every point must have >= 1 observation (Tracking.cc:1858 drops the others before the CRF).
 * kf_ptr (optional, [B+1]): problem b only references keyframes [kf_ptr[b], kf_ptr[b+1]) -- lets the unary kernel
 * keep the current problem's keyframe table in shared memory; obs_kf stays a global keyframe index. */
int lccrf_frames_set_map_inputs(lccrf_frames *fr, const float *xyz, const int *obs_ptr, const int *obs_kf,
                                const float *obs_uv, int nKF, const float *kf_pose, const float *kf_intr,
                                const float *kf_bounds, const float *kp2d, const int *kf_ptr);
/* device-resident run of the whole batch, asynchronous on the context's stream */
int lccrf_frames_run(lccrf_frames *fr);
/* copy results back (synchronises): map [NT] (0 = moving, 1 = static), prob [NT*2]; either may be NULL */
int lccrf_frames_get_outputs(lccrf_frames *fr, short *map, float *prob);
/* Pipelined end-to-end submission, depth 2.  One call = one step through host buffers: the step's inputs go up on a
 * dedicated copy stream into input slot `slot` (0 or 1), the batch runs on the context's stream as soon as they have
 * landed, and map [NT] / prob [NT*2] (either may be NULL) come back into the caller's buffers.  The call returns
 * without waiting; lccrf_frames_wait(fr, slot) blocks until that submission's outputs are in host memory.  Alternating
 * the two slots overlaps the upload of step i+1 with the compute of step i.  Host buffers should be pinned and must
 * stay valid until the matching wait.
 * submit_map: map-snapshot inputs (lccrf_frames_set_map_inputs layout); obs_kf holds int32 (obs_kf_bytes = 4) or
 * uint16 (obs_kf_bytes = 2, nKF <= 65536) keyframe indices.  submit: direct per-frame vectors (set_inputs layout). */
int lccrf_frames_submit_map(lccrf_frames *fr, int slot, const float *xyz, const int *obs_ptr, const void *obs_kf,
                            int obs_kf_bytes, const float *obs_uv, int nKF, const float *kf_pose, const float *kf_intr,
                            const float *kf_bounds, const float *kp2d, const int *kf_ptr, short *map_out,
                            float *prob_out);
/* Resident keyframe keypoints + indexed observations.  In the reference an observation is the pair
 * (KeyFrame*, feature index) of MapPoint::mObservations (std::map<KeyFrame*, size_t>, include/MapPoint.h:115); the
 * observed keypoint is looked up as pKF->mvKeysUn[idx].pt (src/Tracking.cc:1831), a per-keyframe array that never
 * changes once the keyframe exists (include/KeyFrame.h:164).  This entry keeps those arrays resident in HBM:
 * keyframes [kf_first, kf_first + kf_count) get kp_uv [kf_count][stride][2] (undistorted keypoints, rows padded to
 * `stride` = the extractor's feature budget); the table grows as keyframes are inserted, earlier rows stay.
 * Synchronises; not to be called while a submission is in flight. */
int lccrf_frames_set_keyframe_keypoints(lccrf_frames *fr, int kf_first, int kf_count, int stride, const float *kp_uv);
/* lccrf_frames_set_map_inputs / lccrf_frames_submit_map with indexed observations: obs_ref [nnz][2] holds
 * {keyframe index, feature index} as uint16 pairs (index_bytes = 2: nKF and stride <= 65536) or int32 pairs
 * (index_bytes = 4); the keypoint of observation e is kp_table[obs_ref[e].kf][obs_ref[e].fid].  4 instead of 10 bytes
 * per observation cross PCIe.  Feature indices must be < stride (not checked: host-side O(nnz) work). */
int lccrf_frames_set_map_inputs_indexed(lccrf_frames *fr, const float *xyz, const int *obs_ptr, const void *obs_ref,
                                        int index_bytes, int nKF, const float *kf_pose, const float *kf_intr,
                                        const float *kf_bounds, const float *kp2d, const int *kf_ptr);
int lccrf_frames_submit_map_indexed(lccrf_frames *fr, int slot, const float *xyz, const int *obs_ptr, const void *obs_ref,
                                    int index_bytes, int nKF, const float *kf_pose, const float *kf_intr,
                                    const float *kf_bounds, const float *kp2d, const int *kf_ptr, short *map_out,
                                    float *prob_out);
int lccrf_frames_submit(lccrf_frames *fr, int slot, const float *observs, const float *error, const float *depth,
                        const float *kp2d, short *map_out, float *prob_out);
int lccrf_frames_wait(lccrf_frames *fr, int slot);
/* Label application, the hand-off after inference: replaces the scan of res_label in
 *   Tracking::DynamicDetectionWithCRF   src/Tracking.cc:1945-1955
 *     for (i < N) if (res_label[i] == 0) { maps.erase(fid); pMP->SetBadFlag(); mvpMapPoints[fid] = NULL; }
 * by a stable partition of the batch's MAP labels computed on the device: dyn_list holds, problem after problem and
 * in point order, the points labelled moving (label 0) -- exactly the elements the reference loop acts on, in its
 * order -- and stat_list the survivors (label 1) that the second PoseOptimization (Tracking.cc:1002) keeps.
 * Problem b owns dyn_list[dyn_ptr[b] .. dyn_ptr[b+1]) and stat_list[stat_ptr[b] .. stat_ptr[b+1]).  An element is
 * fid[i] (featureMapAssos[i].fid, [NT]) when fid is given, else the point's index inside its problem.
 * dyn_ptr / stat_ptr: [B+1]; dyn_list / stat_list: [NT] (only the first dyn_ptr[B] / stat_ptr[B] entries are
 * written).  Any output may be NULL.  Valid after lccrf_frames_run / lccrf_frames_wait; synchronises. */
int lccrf_frames_partition(lccrf_frames *fr, const int *fid, int *dyn_ptr, int *dyn_list, int *stat_ptr,
                           int *stat_list);
/* diagnostics: init labels [NT], unary-derived vectors, per-problem lattice sizes [B*2] */
int lccrf_frames_get_debug(lccrf_frames *fr, short *init_label, float *observs, float *error, float *depth,
                           int *V);
/* diagnostics of lattice set k (0 = appearance, 1 = smoothness) after a run: out8 = {#long rows, #chunks, #pieces,
 * compose tickets, chunk records applied in O(1), crossing windows applied, chunks summed for real, zero chunks}
 * (the last four accumulate over the filter calls since the lattice was built) */
int lccrf_frames_debug_counters(lccrf_frames *fr, int k, int *out8);
/* algorithmic bytes of one lccrf_frames_run by the SURVEY 8(d) formulas with the actual V (valid after a run) */
int lccrf_frames_algorithmic_bytes(lccrf_frames *fr, double *total, double *per_iteration, double *unary);

/* ---------------------------------------------------------------- batched images --------- */
/* B independent full-image CRFs in one launch sequence: for every image
 *   DenseCRFCPU<M> crf(W*H); crf.setUnaryEnergy(...) or setUnaryEnergyFromLabel(...);
 *   crf.addPairwiseEnergy(PottsPotentialCPU<M,F>::FromImage(W, H, w, posdev, img, featuredev)) for each kernel;
 *   crf.inference(n_iterations, true, relax)
 *   (Thirdparty/DenseCRF/examples/example_cpu.cpp:80-102).  Image sizes, labels and kernels are fixed at create; each
 * run rebuilds the lattices from the current pixels.  Marginals and MAP labels are bit-identical, image by image, to the
 * lccrf_crf path (lccrf_crf_add_potts_image) on the same inputs. */
typedef struct lccrf_images lccrf_images;
/* one Potts potential of PottsPotentialCPU<M,F>::FromImage (pairwise_cpu.h:34-50) */
typedef struct lccrf_image_kernel {
    int F;              /* 2: Gaussian on (x/posdev, y/posdev); C + 2: bilateral, adds the C image channels / featuredev */
    float w, posdev, featuredev;
} lccrf_image_kernel;
/* B images; image b is W[b] x H[b] pixels, row-major (pixel index y*W[b] + x, as pairwise_cpu.h:41-44), images
 * concatenated in order (NT = sum of W[b]*H[b] pixels).  C channels per pixel (0 when every kernel has F == 2), L labels,
 * K kernels in the order addPairwiseEnergy would attach them.  At most 2^22 pixels per image. */
int  lccrf_images_create(lccrf_ctx *ctx, int B, const int *W, const int *H, int C, int L, int K,
                         const lccrf_image_kernel *kernels, lccrf_images **out);
void lccrf_images_destroy(lccrf_images *im);
/* img [NT*C] u8 (img_is_u8) or f32, NULL when C == 0 or no kernel is bilateral.  unary [NT*L]: setUnaryEnergy
 * (densecrf3d.h:41-43).  The arrays have been read when the call returns (it synchronises). */
int  lccrf_images_set_inputs(lccrf_images *im, const void *img, int img_is_u8, const float *unary);
/* ... or setUnaryEnergyFromLabel (densecrf3d.h:108-130): label [NT] in [-1, L), tables as lccrf_crf_set_unary_from_label.
 * Labels are checked on the device: one outside [-1, L) makes lccrf_images_get_outputs return LCCRF_ERR_ARG. */
int  lccrf_images_set_inputs_from_label(lccrf_images *im, const void *img, int img_is_u8, const short *label,
                                        float u_energy, const float *n_energies, const float *p_energies);
/* inference(n_iterations, true, relax) for every image, asynchronous on the context's stream.  With option "graphs" the
 * second run of the same (n_iterations, relax, input mode) captures a CUDA graph and later runs replay it. */
int  lccrf_images_run(lccrf_images *im, int n_iterations, float relax);
/* synchronises; map [NT], prob [NT*L], either may be NULL; reports errors raised on the device (key range, labels).
 * LCCRF_ERR_STATE before the first run.  The object stays usable after an error. */
int  lccrf_images_get_outputs(lccrf_images *im, short *map, float *prob);
/* M_ of every lattice after a run: V [B*K], image-major (diagnostics / tests); synchronises */
int  lccrf_images_vertices(lccrf_images *im, int *V);

/* ---------------------------------------------------------------- device-resident map ----- */
/* In the reference the observation lists, keyframe poses and keypoints are persistent MAP state that tracking only reads
 * (Tracking::ComputeMapPointErrAndObserv, src/Tracking.cc:1803-1839) and local mapping mutates a little per keyframe.
 * lccrf_map keeps that state in HBM, so that per frame only the list of visible map points, the frame's keypoints and the
 * step's changes cross PCIe.  One lccrf_map_delta carries the changes of one step; every member mirrors a reference
 * mutator (counts of 0 / NULL arrays = nothing to do):
 *   kf_*      new keyframes [kf_first, kf_first + kf_count)   KeyFrame ctor + Map::AddKeyFrame (src/Map.cc:32-38):
 *             pose rows [Rcw|tcw] (12), fx fy cx cy, mnMinX mnMaxX mnMinY mnMaxY, and mvKeysUn as [kp_stride][2] rows
 *             (include/KeyFrame.h:157,164,185-188).  Ids are the caller's dense indices; re-sending an id overwrites it.
 *   pose      KeyFrame::SetPose (src/KeyFrame.cc:70-86; bundle adjustment, loop closing): pose_kf [n_pose] ids (NULL =
 *             keyframes 0..n_pose-1), pose [n_pose*12]
 *   xyz       MapPoint ctor / MapPoint::SetWorldPos (src/MapPoint.cc:73-78): xyz_id [n_xyz] (NULL = points 0..n_xyz-1)
 *   erase     MapPoint::EraseObservation(pKF) (src/MapPoint.cc:111-141): removes the observation of point erase_pt[i] in
 *             keyframe erase_kf[i] (no-op when absent, as :116); the rest of the list keeps its order
 *   bad       MapPoint::SetBadFlag (src/MapPoint.cc:151-168, called for moving points at Tracking.cc:1952): the point
 *             loses all observations
 *   add       MapPoint::AddObservation(pKF, idx) (src/MapPoint.cc:98-109): appends (add_kf[i], add_fid[i]) to point
 *             add_pt[i] unless the point already has an observation in that keyframe (:101-102); the observed keypoint mvKeysUn[idx].pt is looked up in the resident keyframe once, here
 * Applied in exactly this order.  Within one SEGMENT of the erase / add lists (the whole list unless *_seg_ptr says
 * otherwise) a point may appear at most once: one keyframe inserts / culls at most one observation per point.  A
 * repetition is detected on the device and reported as LCCRF_ERR_ARG by the call that synchronises.  Observation order
 * = insertion order (the reference iterates a std::map<KeyFrame*, size_t>, i.e. pointer order, which no restatement can
 * reproduce); a map filled through lccrf_map_set_observations / deltas gives bit-identical results to the same lists
 * passed to lccrf_frames_set_map_inputs. */
typedef struct lccrf_map lccrf_map;
typedef struct lccrf_map_delta {
    int kf_first, kf_count;
    const float *kf_pose, *kf_intr, *kf_bounds, *kf_keypoints;
    int n_pose;
    const int *pose_kf;
    const float *pose;
    int n_xyz;
    const int *xyz_id;
    const float *xyz;
    int n_erase;
    const int *erase_pt, *erase_kf;
    int n_bad;
    const int *bad_pt;
    int n_add;
    const int *add_pt, *add_kf, *add_fid;
    /* optional segmentation of the erase / add lists (host arrays [n_*_seg + 1], first 0, last n_erase / n_add): one
     * segment per culled / inserted keyframe, applied one after the other, so that a step may carry several keyframes
     * that touch the same point; the once-per-point rule then holds per segment.  0 / NULL = one segment. */
    int n_erase_seg;
    const int *erase_seg_ptr;
    int n_add_seg;
    const int *add_seg_ptr;
} lccrf_map_delta;
/* kp_stride: keypoint slots per keyframe (the ORB extractor's feature budget, ORBextractor.nFeatures) */
int lccrf_map_create(lccrf_ctx *ctx, int kp_stride, lccrf_map **out);
void lccrf_map_destroy(lccrf_map *map);
/* apply one delta; synchronises, so the host arrays may be reused on return */
int lccrf_map_apply(lccrf_map *map, const lccrf_map_delta *delta);
/* bulk load (a map read from disk, a replay start): replaces the observation lists of points [pt_first, pt_first+count)
 * by the CSR obs_ptr [count+1] / obs_ref [nnz][2] = {keyframe, feature index}; lists keep CSR order.  The keyframes must
 * exist.  Synchronises. */
int lccrf_map_set_observations(lccrf_map *map, int pt_first, int count, const int *obs_ptr, const int *obs_ref);
/* room for `entries` more observations (the pool also grows on its own, by doubling, ahead of demand) */
int lccrf_map_reserve_observations(lccrf_map *map, long long entries);
/* keyframes, map points (highest id + 1), live observations, pool entries in use (incl. abandoned runs), pool capacity */
int lccrf_map_sizes(lccrf_map *map, int *n_kf, int *n_points, long long *n_obs, long long *pool_used, long long *pool_cap);
/* read back the observation lists of n points in the lccrf_frames_set_map_inputs layout (tests, snapshot files):
 * obs_ptr [n+1]; obs_kf / obs_uv hold up to `cap` observations (LCCRF_ERR_ARG when more are needed; obs_ptr[n] tells).
 * xyz [n*3] optional.  Synchronises. */
int lccrf_map_export(lccrf_map *map, int n, const int *point_id, int *obs_ptr, int *obs_kf, float *obs_uv, long long cap,
                     float *xyz);

/* Frame batch against the resident map: problem b's points are the map points point_id[prob_ptr[b] .. prob_ptr[b+1])
 * (mCurrentFrame.mvpMapPoints[i] of the matched features, Tracking.cc:1849-1870; every one needs >= 1 observation,
 * :1858), kp2d [NT*2] their keypoints in the frame.  `delta` (optional) is applied first.  kf_ptr as in
 * lccrf_frames_set_map_inputs.  set_visible uploads on the context's stream (follow with lccrf_frames_run);
 * submit_visible is the pipelined form (slot 0 / 1, uploads on the copy stream, results into map_out / prob_out, finish
 * with lccrf_frames_wait): host arrays, including the delta's, must stay valid until that wait returns.  Both equal
 * lccrf_frames_set_visible_maps / submit_visible_maps with the one map {map}, map_prob {0, B} and deltas = delta. */
int lccrf_frames_set_visible(lccrf_frames *fr, lccrf_map *map, const lccrf_map_delta *delta, const int *point_id,
                             const float *kp2d, const int *kf_ptr);
int lccrf_frames_submit_visible(lccrf_frames *fr, int slot, lccrf_map *map, const lccrf_map_delta *delta,
                                const int *point_id, const float *kp2d, const int *kf_ptr, short *map_out, float *prob_out);
/* Frame batch against several resident maps (several tracked sequences on one GPU): map m serves problems
 * [map_prob[m], map_prob[m+1]) (map_prob [n_maps+1], first 0, last B, non-decreasing; a map may serve no problem and
 * still carry a delta).  point_id [NT] names points of the problem's own map; kf_ptr (optional, [B+1]) slices in the
 * problem's own map's keyframe indices: within a map's segment it starts at 0 and does not decrease, the segment's last
 * problem ends at that map's keyframe count, and kf_ptr[B] is the keyframe count of the last problem's map.  deltas:
 * NULL or [n_maps] (a zeroed delta = nothing to do), deltas[m] applied to maps[m] first.  Every map belongs to fr's
 * context and appears once.  Per problem the results are bit-identical to lccrf_frames_set_visible on that problem's
 * map.  Same lifetime rules as set_visible / submit_visible. */
int lccrf_frames_set_visible_maps(lccrf_frames *fr, int n_maps, lccrf_map *const *maps, const lccrf_map_delta *deltas,
                                  const int *map_prob, const int *point_id, const float *kp2d, const int *kf_ptr);
int lccrf_frames_submit_visible_maps(lccrf_frames *fr, int slot, int n_maps, lccrf_map *const *maps,
                                     const lccrf_map_delta *deltas, const int *map_prob, const int *point_id,
                                     const float *kp2d, const int *kf_ptr, short *map_out, float *prob_out);
/* Epipolar prior of the next run / submission of `slot` (RroughClassify's second branch, Tracking.cc:2001-2010):
 * p4 [NT] = mvFeatureMatchProb[fid] of every point (0.0 without a match, :2003); has_prior [B] (optional) = 0 for the
 * problems whose frame had no fundamental matrix (mvFeatureMatchProb.empty(), :1994) -- those take the first branch.
 * p4 == NULL clears the prior.  The arrays are read when the slot's inputs are uploaded (same lifetime rule). */
int lccrf_frames_set_prior(lccrf_frames *fr, int slot, const double *p4, const unsigned char *has_prior);
/* Label-application lists of a pipelined submission: registers host buffers that lccrf_frames_submit_* fills for `slot`
 * (lccrf_frames_partition semantics; dyn_list / stat_list [NT] each, dyn_ptr / stat_ptr [B+1], fid [NT] optional);
 * valid after lccrf_frames_wait(slot).  All NULL unregisters. */
int lccrf_frames_set_partition_outputs(lccrf_frames *fr, int slot, const int *fid, int *dyn_ptr, int *dyn_list, int *stat_ptr,
                                       int *stat_list);

/* ---------------------------------------------------------------- snapshot / replay files - */
/* CRF-input snapshot format (SURVEY 8f row 1; host-only, no device needed).  A file holds, frame after frame, the flat
 * restatement of what Tracking::DynamicDetectionWithCRF gathers (src/Tracking.cc:1849-1870) and what
 * ComputeMapPointErrAndObserv dereferences (:1803-1839) -- the lccrf_frames_set_map_inputs layout plus the feature
 * id of every point (featureMapAssos[i].fid) -- so a TUM/Bonn sequence can be replayed through the CRF without
 * ORB-SLAM.  Byte layout: lc-crf-slam_b200/csrc/snapshot.cu.  Records are appended and individually checksummed; a
 * file cut off by a crash still yields every complete frame (lccrf_snapshot_truncated tells). */
typedef struct lccrf_snapshot_writer lccrf_snapshot_writer;
typedef struct lccrf_snapshot_reader lccrf_snapshot_reader;
typedef struct lccrf_snapshot_info {
    int N, nKF;
    long long nnz;
    long long frame_id;  /* mCurrentFrame.mnId */
    double timestamp;
    int stored_kf_bytes; /* 2: keyframe indices stored as uint16 (nKF <= 65536), 4: int32 */
} lccrf_snapshot_info;
/* append != 0 continues an existing file (created when missing) */
int lccrf_snapshot_writer_open(const char *path, int append, lccrf_snapshot_writer **out);
/* one frame; arrays as in lccrf_map_point_unary, kp2d [N*2], fid [N] (NULL = 0..N-1).  Validates the CSR. */
int lccrf_snapshot_write_frame(lccrf_snapshot_writer *w, long long frame_id, double timestamp, int N, const float *xyz,
                               const int *obs_ptr, const int *obs_kf, const float *obs_uv, int nKF, const float *kf_pose,
                               const float *kf_intr, const float *kf_bounds, const float *kp2d, const int *fid);
int lccrf_snapshot_writer_close(lccrf_snapshot_writer *w);
int lccrf_snapshot_reader_open(const char *path, lccrf_snapshot_reader **out);
void lccrf_snapshot_reader_close(lccrf_snapshot_reader *r);
int lccrf_snapshot_num_frames(const lccrf_snapshot_reader *r);
int lccrf_snapshot_truncated(const lccrf_snapshot_reader *r);
int lccrf_snapshot_frame_info(const lccrf_snapshot_reader *r, int i, lccrf_snapshot_info *info);
/* read frame i into caller buffers sized from frame_info (any pointer may be NULL); obs_kf comes back as int32
 * (obs_kf_bytes = 4) or uint16 (2, what lccrf_frames_submit_map takes).  Verifies the checksum and the structure
 * (CSR monotone, keyframe indices in range) and fails with LCCRF_ERR_STATE on a corrupt frame. */
int lccrf_snapshot_read_frame(lccrf_snapshot_reader *r, int i, float *xyz, int *obs_ptr, void *obs_kf, int obs_kf_bytes,
                              float *obs_uv, float *kf_pose, float *kf_intr, float *kf_bounds, float *kp2d, int *fid);

#ifdef __cplusplus
}
#endif
#endif /* LCCRF_H */
