/* images_batch.c -- the batched image CRF (include/lccrf.h, "batched images") from plain C: three images of different
 * sizes, a Gaussian and a bilateral kernel on an RGB image (the recipe of example_cpu.cpp:80-102), labels with 2/3
 * unknown, ten mean-field iterations, MAP labels and marginals of every image.  Runs the batch twice with new labels to
 * show that the object is reused.  Exits 2 when no device is usable (there is no CPU fallback). */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "lccrf.h"

#define CHECK(call)                                                                      \
    do {                                                                                 \
        int rc_ = (call);                                                                \
        if (rc_ != LCCRF_OK) {                                                           \
            fprintf(stderr, "%s failed (%d): %s\n", #call, rc_, lccrf_last_error());     \
            return 1;                                                                    \
        }                                                                                \
    } while (0)

enum { B = 3, C = 3, L = 2, K = 2 };

int main(void) {
    const int W[B] = {64, 33, 40}, H[B] = {48, 17, 30};
    const lccrf_image_kernel kernels[K] = {{2, 3.0f, 3.0f, 0.0f}, {C + 2, 10.0f, 60.0f, 20.0f}};
    lccrf_ctx *ctx = NULL;
    lccrf_images *im = NULL;
    int b, i, NT = 0, run, V[B * K];
    if (lccrf_ctx_create(0, &ctx) != LCCRF_OK) {
        fprintf(stderr, "%s\n", lccrf_last_error());
        return 2;
    }
    for (b = 0; b < B; b++) NT += W[b] * H[b];
    unsigned char *img = malloc((size_t)NT * C);
    short *label = malloc((size_t)NT * sizeof(short)), *map = malloc((size_t)NT * sizeof(short));
    float *prob = malloc((size_t)NT * L * sizeof(float));
    if (!img || !label || !map || !prob) return 1;
    /* a bright disc on a dark background in every image */
    for (b = 0, i = 0; b < B; b++) {
        int x, y;
        for (y = 0; y < H[b]; y++)
            for (x = 0; x < W[b]; x++, i++) {
                const float dx = x - 0.5f * W[b], dy = y - 0.5f * H[b];
                const int fg = dx * dx + dy * dy < 0.1f * W[b] * H[b];
                img[3 * i] = (unsigned char)(fg ? 200 : 60);
                img[3 * i + 1] = (unsigned char)(fg ? 80 : 120 + (x * 7 + y * 3) % 9);
                img[3 * i + 2] = (unsigned char)(fg ? 60 : 180);
            }
    }
    /* setUnaryEnergyFromLabel's tables for one confidence c (densecrf3d.h:109-114) */
    const float c = 0.7f;
    const float u_en = -logf(1.0f / L), n_en[L] = {-logf((1.0f - c) / (L - 1)), -logf((1.0f - c) / (L - 1))},
                p_en[L] = {-logf(c), -logf(c)};
    CHECK(lccrf_images_create(ctx, B, W, H, C, L, K, kernels, &im));
    for (run = 0; run < 2; run++) {
        for (b = 0, i = 0; b < B; b++) {
            int x, y;
            for (y = 0; y < H[b]; y++)
                for (x = 0; x < W[b]; x++, i++) {
                    const int fg = img[3 * i] == 200;
                    label[i] = (short)((i + run) % 3 == 0 ? fg : -1);  /* 2/3 of the pixels unknown */
                }
        }
        CHECK(lccrf_images_set_inputs_from_label(im, img, 1, label, u_en, n_en, p_en));
        CHECK(lccrf_images_run(im, 10, 1.0f));
        CHECK(lccrf_images_get_outputs(im, map, prob));
        for (b = 0, i = 0; b < B; b++) {
            int fg_right = 0, n = W[b] * H[b], j;
            for (j = 0; j < n; j++, i++) {
                const float s = prob[2 * i] + prob[2 * i + 1];
                if (map[i] < 0 || map[i] >= L || !(fabsf(s - 1.0f) < 1e-5f)) {
                    fprintf(stderr, "image %d pixel %d: map %d, marginals sum to %g\n", b, j, map[i], s);
                    return 1;
                }
                fg_right += map[i] == (img[3 * i] == 200);
            }
            printf("run %d image %d (%dx%d): %.1f%% of the pixels labelled disc / background correctly\n", run, b, W[b], H[b],
                   100.0 * fg_right / n);
            if (fg_right < n * 8 / 10) return 1;
        }
    }
    CHECK(lccrf_images_vertices(im, V));
    for (b = 0; b < B; b++) printf("image %d: lattices of %d and %d vertices\n", b, V[b * K], V[b * K + 1]);
    lccrf_images_destroy(im);
    lccrf_ctx_destroy(ctx);
    free(img);
    free(label);
    free(map);
    free(prob);
    return 0;
}
