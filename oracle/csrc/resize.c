/* Oracle restatement of cv2.resize(src, (W, H), interpolation=cv2.INTER_LINEAR) for float32 planes with h, w >= 2,
 * as the opencv-python 4.13.0 wheel computes it with its IPP HAL on (the default).  Per axis with n_in source and
 * n_out output pixels, output index d:
 *
 *   f = (d + 0.5) * (n_in / n_out) - 0.5        fp64, every step rounded on its own
 *   s = floor(f), a = (float)(f - s)            the fraction rounded to fp32 from the fp64 value
 *   s1 = s + 1
 *   s < 0 or s >= n_in - 1: a BORDER tap, s and s1 clamped to the nearest source index
 *
 * Horizontal pass first, then the vertical pass, each with one fp32 subtract and ONE fp32 fma (libm fmaf, a single
 * rounding; an fp32 fma emulated in fp64 would round twice):
 *
 *   R[y][X]   = border x ? S[y][s0x] : fmaf(S[y][s1x] - S[y][s0x], ax, S[y][s0x])
 *   out[Y][X] = fmaf(R[s1y][X] - R[s0y][X], ay, R[s0y][X])          interior y
 *             = R[s0y][X]                                            border y, interior x
 *             = fmaf(R[s0y][X] - R[s0y][X], 0, R[s0y][X])            border y and border x (the four corner blocks)
 *
 * The border cases only matter for non-finite values: a border tap never reads its second source pixel (an Inf next
 * to the border does not turn the border into NaN), except in the corner blocks, where an Inf becomes NaN.  A shape
 * equal to the source is a copy.  Built with -ffp-contract=off so that the compiler adds no contraction of its own. */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    int s0, s1;
    float a;
} tap_t;

static void taps(int n_in, int n_out, tap_t *t) {
    const double scale = (double)n_in / (double)n_out;
    for (int d = 0; d < n_out; d++) {
        const double f = ((double)d + 0.5) * scale - 0.5;
        const double fl = floor(f);
        int s = (int)fl;
        float a = (float)(f - fl);
        int s1 = s + 1;
        if (s < 0) { s = s1 = 0; a = 0.0f; }
        if (s >= n_in - 1) { s = s1 = n_in - 1; a = 0.0f; }
        t[d].s0 = s;
        t[d].s1 = s1;
        t[d].a = a;
    }
}

/* src [n,h,w] -> dst [n,H,W], float32.  Returns 0, or -2 for a shape the rule does not cover (h or w < 2, or any
 * dimension < 1), -1 when out of memory. */
int oracle_resize_linear_f32(const float *src, int n, int h, int w, float *dst, int H, int W) {
    if (n < 1 || h < 2 || w < 2 || H < 1 || W < 1) return -2;
    if (h == H && w == W) {
        memcpy(dst, src, sizeof(float) * (size_t)n * h * w);
        return 0;
    }
    tap_t *tx = malloc(sizeof(tap_t) * (size_t)W), *ty = malloc(sizeof(tap_t) * (size_t)H);
    float *r0 = malloc(sizeof(float) * (size_t)W), *r1 = malloc(sizeof(float) * (size_t)W);
    if (!tx || !ty || !r0 || !r1) { free(tx); free(ty); free(r0); free(r1); return -1; }
    taps(w, W, tx);
    taps(h, H, ty);
    for (int i = 0; i < n; i++) {
        const float *S = src + (size_t)i * h * w;
        float *O = dst + (size_t)i * H * W;
        for (int Y = 0; Y < H; Y++) {
            const float *a0 = S + (size_t)ty[Y].s0 * w, *a1 = S + (size_t)ty[Y].s1 * w;
            for (int X = 0; X < W; X++) {
                const tap_t t = tx[X];
                r0[X] = t.s0 == t.s1 ? a0[t.s0] : fmaf(a0[t.s1] - a0[t.s0], t.a, a0[t.s0]);
                r1[X] = t.s0 == t.s1 ? a1[t.s0] : fmaf(a1[t.s1] - a1[t.s0], t.a, a1[t.s0]);
            }
            const float ay = ty[Y].a;
            if (ty[Y].s0 == ty[Y].s1)  /* border row: copied, except the corners (see the header) */
                for (int X = 0; X < W; X++)
                    O[(size_t)Y * W + X] = tx[X].s0 == tx[X].s1 ? fmaf(r0[X] - r0[X], 0.0f, r0[X]) : r0[X];
            else
                for (int X = 0; X < W; X++) O[(size_t)Y * W + X] = fmaf(r1[X] - r0[X], ay, r0[X]);
        }
    }
    free(tx); free(ty); free(r0); free(r1);
    return 0;
}
