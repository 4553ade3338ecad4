/*
 * resample_ref.c -- reference of the resampler of scaled distorted frames (include/ssimu2_b200.h, ssimu2_source.width /
 * height), restated on the CPU for tests/test_scaled_sources.py, which builds it with
 * gcc -O2 -fPIC -std=c11 -ffp-contract=off -fno-fast-math (no implicit FMA contraction: fused ops are explicit fmaf()).
 *
 * One plane of nch interleaved channels, upscaled in its own sample domain: separable bicubic Catmull-Rom (Keys,
 * a = -0.5), centre-aligned (sx = (x + 0.5) * in / out - 0.5), clamp-to-edge, taps floor(sx) - 1 .. floor(sx) + 2 in
 * ascending order; weights in double rounded to float; f32 evaluation horizontally first, a = w0*s0 then three fmaf
 * steps, then the same chain vertically over the 4 row results.  u8 / u16 results: round half to even, clamp; f32
 * results: unrounded, unclamped.  Not ffmpeg swscale's bicubic (B = 0, C = 0.6).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

static double keys_weight(double t)
{
    if (t < 1.0) return (1.5 * t - 2.5) * t * t + 1.0;
    if (t < 2.0) return ((-0.5 * t + 2.5) * t - 4.0) * t + 2.0;
    return 0.0;
}

/* Taps of an axis of `in` -> `out` samples: j0[x] = floor(sx) - 1 (unclamped), w[4 * x + k] the weight of tap j0[x] + k. */
void rs_ref_taps(int in, int out, int *j0, float *w)
{
    const double scale = (double)in / (double)out;
    for (int x = 0; x < out; x++) {
        const double sx = (x + 0.5) * scale - 0.5;
        const int i = (int)floor(sx);
        for (int k = 0; k < 4; k++) w[4 * x + k] = (float)keys_weight(fabs(sx - (double)(i - 1 + k)));
        j0[x] = i - 1;
    }
}

static float load(int type, const uint8_t *row, int idx)
{
    if (type == 0) return (float)row[idx];
    if (type == 1) return (float)((const uint16_t *)row)[idx];
    return ((const float *)row)[idx];
}

static int clampi(int v, int lo, int hi) { return v < lo ? lo : v > hi ? hi : v; }

/* One plane of `nch` interleaved channels, each in_w x in_h -> out_w x out_h.  type: 0 = u8, 1 = u16, 2 = f32 samples;
 * pitches in bytes.  Returns 0, or -1 when out of memory. */
int rs_ref_plane(int type, const void *src, size_t src_pitch, int in_w, int in_h, int nch, void *dst, size_t dst_pitch,
                 int out_w, int out_h)
{
    int *jx = malloc(sizeof(int) * out_w), *jy = malloc(sizeof(int) * out_h);
    float *wx = malloc(sizeof(float) * 4 * out_w), *wy = malloc(sizeof(float) * 4 * out_h);
    float *rows = malloc(sizeof(float) * (size_t)in_h * out_w * nch);
    if (!jx || !jy || !wx || !wy || !rows) {
        free(jx); free(jy); free(wx); free(wy); free(rows);
        return -1;
    }
    rs_ref_taps(in_w, out_w, jx, wx);
    rs_ref_taps(in_h, out_h, jy, wy);
    /* horizontal pass of every source row */
    for (int r = 0; r < in_h; r++) {
        const uint8_t *row = (const uint8_t *)src + (size_t)r * src_pitch;
        for (int x = 0; x < out_w; x++)
            for (int c = 0; c < nch; c++) {
                const float *w = wx + 4 * x;
                float a = w[0] * load(type, row, clampi(jx[x], 0, in_w - 1) * nch + c);
                a = fmaf(w[1], load(type, row, clampi(jx[x] + 1, 0, in_w - 1) * nch + c), a);
                a = fmaf(w[2], load(type, row, clampi(jx[x] + 2, 0, in_w - 1) * nch + c), a);
                a = fmaf(w[3], load(type, row, clampi(jx[x] + 3, 0, in_w - 1) * nch + c), a);
                rows[((size_t)r * out_w + x) * nch + c] = a;
            }
    }
    /* vertical pass over the row results */
    for (int y = 0; y < out_h; y++) {
        uint8_t *out = (uint8_t *)dst + (size_t)y * dst_pitch;
        const float *w = wy + 4 * y;
        const float *r0 = rows + (size_t)clampi(jy[y], 0, in_h - 1) * out_w * nch;
        const float *r1 = rows + (size_t)clampi(jy[y] + 1, 0, in_h - 1) * out_w * nch;
        const float *r2 = rows + (size_t)clampi(jy[y] + 2, 0, in_h - 1) * out_w * nch;
        const float *r3 = rows + (size_t)clampi(jy[y] + 3, 0, in_h - 1) * out_w * nch;
        for (int i = 0; i < out_w * nch; i++) {
            float a = w[0] * r0[i];
            a = fmaf(w[1], r1[i], a);
            a = fmaf(w[2], r2[i], a);
            a = fmaf(w[3], r3[i], a);
            if (type == 2) {
                ((float *)out)[i] = a;
            } else {
                const float v = fminf(fmaxf(rintf(a), 0.0f), type == 0 ? 255.0f : 65535.0f);
                if (type == 0) out[i] = (uint8_t)v; else ((uint16_t *)out)[i] = (uint16_t)v;
            }
        }
    }
    free(jx); free(jy); free(wx); free(wy); free(rows);
    return 0;
}
