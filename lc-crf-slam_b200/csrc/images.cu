// images.cu -- lccrf_images: B full-image DenseCRFs in one launch sequence.  Per image this is
//   DenseCRFCPU<M> crf(W*H); crf.setUnaryEnergy / setUnaryEnergyFromLabel;
//   crf.addPairwiseEnergy(PottsPotentialCPU<M,F>::FromImage(...)) per kernel; crf.inference(T, true, relax)
// (Thirdparty/DenseCRF/examples/example_cpu.cpp:80-102), with the images' pixels concatenated into one Batch: one
// feature launch, one lattice build and one filter sequence per kernel serve every image.
#include <climits>
#include <string>
#include <vector>

#include "engine.cuh"

using namespace lccrf;

namespace {

enum InputMode { kNoInputs = 0, kUnary = 1, kLabel = 2 };

// what the launch arguments of a run depend on besides the buffers fixed at create: a change captures a new graph
struct RunShape {
    int T = -1;
    float relax = 0.f;
    int mode = kNoInputs, img_is_u8 = 0;
    float u_energy = 0.f;
    bool operator==(const RunShape &o) const {
        return T == o.T && relax == o.relax && mode == o.mode && img_is_u8 == o.img_is_u8 && u_energy == o.u_energy;
    }
};

}  // namespace

struct lccrf_images {
    Ctx *ctx = nullptr;
    Batch b;
    int C = 0;
    bool needs_img = false;                // some kernel is bilateral (F > 2)
    std::vector<lccrf_image_kernel> kern;
    int *width = nullptr;                  // [B] device: W of every image
    std::vector<float *> feat;             // per kernel [NT*F] device
    void *img = nullptr;                   // [NT*C] u8 or f32 device
    short *label = nullptr;                // [NT] device (label mode)
    float *en = nullptr;                   // n_en[L], p_en[L] device (label mode)
    int mode = kNoInputs, img_is_u8 = 1;
    float u_energy = 0.f;
    bool ran = false;
    RunShape shape;                        // of the captured graph
    GraphReplay graph;
};

static int images_enqueue(lccrf_images *im, int T, float relax) {
    Ctx *ctx = im->ctx;
    Batch &b = im->b;
    const int K = (int)b.lat.size();
    // the K lattices are independent until the first mean-field step: odd kernels build on the aux branch
    if (K > 1) LCCRF_TRY(ctx_fork(ctx));
    for (int k = 0; k < K; k++) {
        AuxScope aux(ctx, K > 1 && (k & 1));
        const lccrf_image_kernel &kn = im->kern[k];
        LCCRF_TRY(feat_image_batch(ctx, im->feat[k], b.NT, b.B, b.prob_ptr, im->width, kn.F, kn.posdev, im->img,
                                   im->img_is_u8, kn.featuredev));
        LCCRF_TRY(lattice_set_build(ctx, b, b.lat[k], im->feat[k]));
        LCCRF_TRY(potts_norm(ctx, b, b.lat[k]));
    }
    if (im->mode == kLabel)
        LCCRF_TRY(mf_unary_from_label(ctx, b.unary, im->label, b.NT, b.L, im->u_energy, im->en, im->en + b.L, ctx->d_status));
    if (K > 1) LCCRF_TRY(ctx_join(ctx));
    // inference(T, true, relax)   densecrf_base.h:65-76
    LCCRF_TRY(mf_start(ctx, b));
    for (int it = 0; it < T; it++) LCCRF_TRY(mf_step(ctx, b, relax));
    return mf_build_map(ctx, b);
}

extern "C" {

int lccrf_images_create(lccrf_ctx *h, int B, const int *W, const int *H, int C, int L, int K,
                        const lccrf_image_kernel *kernels, lccrf_images **out) {
    if (!h || !out || (B > 0 && (!W || !H)) || (K > 0 && !kernels)) return fail(LCCRF_ERR_ARG, "NULL argument");
    *out = nullptr;
    if (B < 0) return fail(LCCRF_ERR_ARG, "B must be >= 0");
    if (C < 0) return fail(LCCRF_ERR_ARG, "C must be >= 0");
    if (L < 1 || L > LCCRF_MAX_L) return fail(LCCRF_ERR_ARG, "L must be in [1, LCCRF_MAX_L]");
    if (K < 0 || K > LCCRF_MAX_K) return fail(LCCRF_ERR_ARG, "K must be in [0, LCCRF_MAX_K]");
    bool needs_img = false;
    for (int k = 0; k < K; k++) {
        const int F = kernels[k].F;
        if (F != 2 && F != C + 2) return fail(LCCRF_ERR_ARG, "kernel F must be 2 (Gaussian) or C + 2 (bilateral)");
        if (F > LCCRF_MAX_D) return fail(LCCRF_ERR_ARG, "kernel F exceeds LCCRF_MAX_D");
        needs_img |= F > 2;
    }
    std::vector<int> pp((size_t)B + 1, 0);
    long long total = 0;
    for (int i = 0; i < B; i++) {
        if (W[i] < 0 || H[i] < 0) return fail(LCCRF_ERR_ARG, "image sizes must be >= 0");
        const long long n = (long long)W[i] * H[i];
        if (n > (1 << 22)) return fail(LCCRF_ERR_ARG, "more than 2^22 pixels in one image (fixed-point splat range)");
        total += n;
        if (total > INT_MAX / 2) return fail(LCCRF_ERR_ARG, "too many pixels in one batch");
        pp[i + 1] = (int)total;
    }
    Ctx *ctx = &h->c;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    auto *im = new lccrf_images();
    im->ctx = ctx;
    im->C = C;
    im->needs_img = needs_img;
    im->kern.assign(kernels, kernels + K);
    int rc = batch_init(ctx, im->b, B, pp.data(), L, true);
    // Image-sized problems do not fit the fused blur's shared memory: one CTA per image would walk its lattice out of
    // global memory on a single SM.  Only batches of small images take the fused blur; all others run the element-parallel
    // passes over the vertices of every image (DESIGN.md "Batched images").
    im->b.fused_blur = im->b.maxN <= kFusedBlurMaxN;
    const size_t n = (size_t)(im->b.NT > 0 ? im->b.NT : 1);
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&im->width, (size_t)(B > 0 ? B : 1) * sizeof(int));
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&im->label, n * sizeof(short));
    if (rc == LCCRF_OK) rc = dev_alloc(ctx, (void **)&im->en, 2 * (size_t)L * sizeof(float));
    if (rc == LCCRF_OK && needs_img) rc = dev_alloc(ctx, &im->img, n * C * sizeof(float));
    for (int k = 0; k < K && rc == LCCRF_OK; k++) {
        im->feat.push_back(nullptr);
        rc = dev_alloc(ctx, (void **)&im->feat.back(), n * kernels[k].F * sizeof(float));
    }
    if (rc == LCCRF_OK && B > 0) {
        cudaError_t e = cudaMemcpyAsync(im->width, W, (size_t)B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(LCCRF_ERR_CUDA, std::string("image widths: ") + cudaGetErrorString(e));
    }
    // an empty batch has nothing to build: runs are no-ops and every lattice has 0 vertices
    for (int k = 0; k < K && rc == LCCRF_OK && im->b.NT > 0; k++) {
        LatticeSet *ls = nullptr;
        rc = lattice_set_create(ctx, im->b, kernels[k].F, kernels[k].w, L, &ls);
        if (rc == LCCRF_OK) im->b.lat.push_back(ls);
    }
    if (rc != LCCRF_OK) {
        lccrf_images_destroy(im);
        return rc;
    }
    *out = im;
    return LCCRF_OK;
}

void lccrf_images_destroy(lccrf_images *im) {
    if (!im) return;
    Ctx *ctx = im->ctx;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    graph_drop(im->graph);
    batch_release(ctx, im->b);
    dev_free(ctx, im->width);
    dev_free(ctx, im->label);
    dev_free(ctx, im->en);
    dev_free(ctx, im->img);
    for (float *f : im->feat) dev_free(ctx, f);
    delete im;
}

// the image part of both input calls (on the context's stream; the caller synchronises)
static int images_upload_img(lccrf_images *im, const void *img, int img_is_u8) {
    const size_t NT = (size_t)im->b.NT;
    if (!im->needs_img || NT == 0) return LCCRF_OK;
    if (!img) return fail(LCCRF_ERR_ARG, "img is NULL but a kernel is bilateral (F > 2)");
    const size_t bytes = NT * im->C * (img_is_u8 ? 1 : sizeof(float));
    LCCRF_CUDA(cudaMemcpyAsync(im->img, img, bytes, cudaMemcpyHostToDevice, im->ctx->stream));
    im->img_is_u8 = img_is_u8 ? 1 : 0;
    return LCCRF_OK;
}

int lccrf_images_set_inputs(lccrf_images *im, const void *img, int img_is_u8, const float *unary) {
    if (!im) return fail(LCCRF_ERR_ARG, "images is NULL");
    const size_t NT = (size_t)im->b.NT;
    if (!unary && NT > 0) return fail(LCCRF_ERR_ARG, "unary is NULL");
    Ctx *ctx = im->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    LCCRF_TRY(images_upload_img(im, img, img_is_u8));
    if (NT) LCCRF_CUDA(cudaMemcpyAsync(im->b.unary, unary, NT * im->b.L * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    im->mode = kUnary;
    return LCCRF_OK;
}

int lccrf_images_set_inputs_from_label(lccrf_images *im, const void *img, int img_is_u8, const short *label,
                                       float u_energy, const float *n_energies, const float *p_energies) {
    if (!im || !n_energies || !p_energies) return fail(LCCRF_ERR_ARG, "NULL argument");
    const size_t NT = (size_t)im->b.NT, L = (size_t)im->b.L;
    if (!label && NT > 0) return fail(LCCRF_ERR_ARG, "label is NULL");
    Ctx *ctx = im->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    LCCRF_TRY(images_upload_img(im, img, img_is_u8));
    if (NT) LCCRF_CUDA(cudaMemcpyAsync(im->label, label, NT * sizeof(short), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaMemcpyAsync(im->en, n_energies, L * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaMemcpyAsync(im->en + L, p_energies, L * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    im->mode = kLabel;
    im->u_energy = u_energy;
    return LCCRF_OK;
}

int lccrf_images_run(lccrf_images *im, int n_iterations, float relax) {
    if (!im) return fail(LCCRF_ERR_ARG, "images is NULL");
    if (n_iterations < 0) return fail(LCCRF_ERR_ARG, "n_iterations < 0");
    if (im->mode == kNoInputs) return fail(LCCRF_ERR_STATE, "lccrf_images_run before lccrf_images_set_inputs");
    Ctx *ctx = im->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    if (im->b.NT > 0) {
        RunShape s;
        s.T = n_iterations;
        s.relax = relax;
        s.mode = im->mode;
        s.img_is_u8 = im->img_is_u8;
        s.u_energy = im->mode == kLabel ? im->u_energy : 0.f;
        if (!(s == im->shape)) {
            graph_drop(im->graph);
            im->shape = s;
        }
        LCCRF_TRY(graph_run(ctx, im->graph, [&] { return images_enqueue(im, n_iterations, relax); }));
    }
    im->ran = true;
    return LCCRF_OK;
}

int lccrf_images_get_outputs(lccrf_images *im, short *map, float *prob) {
    if (!im) return fail(LCCRF_ERR_ARG, "images is NULL");
    if (!im->ran) return fail(LCCRF_ERR_STATE, "lccrf_images_get_outputs before lccrf_images_run");
    Ctx *ctx = im->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)im->b.NT;
    if (n && map) LCCRF_CUDA(cudaMemcpyAsync(map, im->b.map, n * sizeof(short), cudaMemcpyDeviceToHost, ctx->stream));
    if (n && prob) LCCRF_CUDA(cudaMemcpyAsync(prob, im->b.cur, n * im->b.L * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    return check_status(ctx);
}

int lccrf_images_vertices(lccrf_images *im, int *V) {
    if (!im || !V) return fail(LCCRF_ERR_ARG, "NULL argument");
    if (!im->ran) return fail(LCCRF_ERR_STATE, "lccrf_images_vertices before lccrf_images_run");
    Ctx *ctx = im->ctx;
    LCCRF_CUDA(cudaSetDevice(ctx->device));
    const int B = im->b.B, K = (int)im->kern.size();
    std::vector<int> vb((size_t)(B + 1) * K, 0);
    for (int k = 0; k < (int)im->b.lat.size(); k++)
        LCCRF_CUDA(cudaMemcpyAsync(vb.data() + (size_t)k * (B + 1), im->b.lat[k]->vbase, (size_t)(B + 1) * sizeof(int),
                                   cudaMemcpyDeviceToHost, ctx->stream));
    LCCRF_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < B; i++)
        for (int k = 0; k < K; k++) V[(size_t)i * K + k] = vb[(size_t)k * (B + 1) + i + 1] - vb[(size_t)k * (B + 1) + i];
    return LCCRF_OK;
}

}  // extern "C"
