/*
 * ssimu2_oracle.c -- CPU restatement of the reference's SSIMULACRA2 frame-pair path.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it.  The product path
 * (turbo_metrics_b200 + libssimu2_b200.so) never links, imports or calls anything here.
 *
 * Parity status: PARITY UNPINNED BY REFERENCE FIXTURES.  The reference ships no golden
 * vectors for this path (its only known answer, 17.398505 +- 0.25 in
 * crates/ssimulacra2-cuda/examples/compare.rs:70-74, is for an image pair that is not in
 * the repository) and its Rust toolchain is absent here, so the reference itself cannot
 * be run.  What IS pinned (tests/test_oracle_constants.py): the sRGB LUT (all 256 entries
 * equal cpu.rs:20-277), the recursive-Gaussian constants (cpu.rs:931-948, re-derived from
 * ssimulacra2-cuda-kernel/build.rs:28-145), the opsin constants, WEIGHT[108], the final
 * polynomial, and "identical images -> 100.0".
 * Independent witnesses (tests/test_oracle_independent.py, no shared code): an exact-FIR float64 model agrees
 * on the score to <= 0.07 on the small golden cases and 0.25 at 1080p; a float32 model with the recursive
 * filter written from the published recurrences is BIT-equal on the filter and within 0.02 on the score at
 * every size, i.e. the gap to the f64 model is the algorithm's own f32 round-off, not a port defect.
 * "Bit-exact" claims of the CUDA path are relative to THIS oracle built with gcc against the libm of this
 * image (glibc 2.39, x86-64, FMA ifunc variants of powf / cbrtf): Rust's f32::cbrt / powf call the platform
 * libm, so another platform's reference run may differ from both in the last bit of those two functions.
 *
 * What it follows (paths relative to /root/reference/crates):
 *   ssimulacra2-cuda/examples/cpu.rs                 the repository's CPU SSIMULACRA2
 *   cuda-colorspace-kernel/src/{biplanar,lib,constants,const_algebra}.rs
 *                                                   NV12 / P016 -> linear RGB (GPU-only in the
 *                                                   reference; restated with libm powf in place
 *                                                   of __nv_fast_powf)
 *   cuda-colorspace-kernel/src/srgb.rs              sRGB u16 / f32 -> linear (same remark)
 *
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math (see oracle/Makefile).  Every fused
 * multiply-add below is an explicit fmaf()/fma() exactly where the Rust source says
 * mul_add; everything else is a separately rounded IEEE operation.
 *
 * Images are planar f32: plane c of a WxH image is p[c*W*H + y*W + x].  The reference
 * uses packed [f32;3] pixels; the layout does not change any arithmetic.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NUM_SCALES 6 /* cpu.rs:11 */

/* ------------------------------------------------------------------------------------ */
/* sRGB 8-bit -> linear.  cpu.rs:20-277 is a 256-entry table; it is reproduced bit for   */
/* bit by v = i * (1/255) [f32]; v <= 0.04045 ? v/12.92 : powf((v+0.055)/1.055, 2.4),    */
/* all in f32 (verified against the reference table in tests/test_oracle_constants.py).  */
/* ------------------------------------------------------------------------------------ */
static float g_srgb8_lut[256];
static int g_srgb8_lut_ready = 0;

static void srgb8_lut_init(void)
{
    if (g_srgb8_lut_ready)
        return;
    const float inv255 = 1.0f / 255.0f;
    for (int i = 0; i < 256; i++) {
        float v = (float)i * inv255;
        float r;
        if (v <= 0.04045f)
            r = v / 12.92f;
        else
            r = powf((v + 0.055f) / 1.055f, 2.4f);
        g_srgb8_lut[i] = r;
    }
    g_srgb8_lut_ready = 1;
}

void oracle_srgb8_lut(float out[256])
{
    srgb8_lut_init();
    memcpy(out, g_srgb8_lut, sizeof(g_srgb8_lut));
}

/* CpuImg::from_srgb, cpu.rs:280-296.  src is packed RGB8 with a row pitch in bytes. */
void oracle_linear_from_srgb8(const uint8_t *src, size_t pitch, int w, int h, float *out)
{
    srgb8_lut_init();
    size_t n = (size_t)w * h;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            for (int c = 0; c < 3; c++)
                out[c * n + (size_t)y * w + x] = g_srgb8_lut[src[y * pitch + 3 * x + c]];
}

/* srgb_inverse_oetf, cuda-colorspace-kernel/src/srgb.rs:40-48 (powf_fast -> powf). */
static float srgb_inverse_oetf(float x)
{
    const float SRGB_ALPHA = 1.0550107f;
    const float SRGB_BETA = 0.0030412825f;
    if (x < 12.92f * SRGB_BETA)
        return x / 12.92f;
    return powf((x + (SRGB_ALPHA - 1.0f)) / SRGB_ALPHA, 2.4f);
}

/* srgb_to_linear::<16>, srgb.rs:68-86 + Sample::conv_to_f lib.rs:19-21 (v / 65535). */
void oracle_linear_from_srgb16(const uint16_t *src, size_t pitch, int w, int h, float *out)
{
    size_t n = (size_t)w * h;
    for (int y = 0; y < h; y++) {
        const uint16_t *row = (const uint16_t *)((const uint8_t *)src + y * pitch);
        for (int x = 0; x < w; x++)
            for (int c = 0; c < 3; c++)
                out[c * n + (size_t)y * w + x] =
                    srgb_inverse_oetf((float)row[3 * x + c] / (float)65535u);
    }
}

/* srgb_to_linear_f32, srgb.rs:112-127. */
void oracle_linear_from_srgbf32(const float *src, size_t pitch, int w, int h, float *out)
{
    size_t n = (size_t)w * h;
    for (int y = 0; y < h; y++) {
        const float *row = (const float *)((const uint8_t *)src + y * pitch);
        for (int x = 0; x < w; x++)
            for (int c = 0; c < 3; c++)
                out[c * n + (size_t)y * w + x] = srgb_inverse_oetf(row[3 * x + c]);
    }
}

/* CpuImg::from_planes route (cpu.rs:298-313): packed linear f32 -> planar, no arithmetic. */
void oracle_linear_from_linearf32(const float *src, size_t pitch, int w, int h, float *out)
{
    size_t n = (size_t)w * h;
    for (int y = 0; y < h; y++) {
        const float *row = (const float *)((const uint8_t *)src + y * pitch);
        for (int x = 0; x < w; x++)
            for (int c = 0; c < 3; c++)
                out[c * n + (size_t)y * w + x] = row[3 * x + c];
    }
}

/* ------------------------------------------------------------------------------------ */
/* NV12 / P016 -> linear RGB.  cuda-colorspace-kernel/src/biplanar.rs:7-70.              */
/* ------------------------------------------------------------------------------------ */
typedef struct { float x, y; } v2;
typedef struct { float x, y, z; } v3;

/* const_algebra.rs:29-31 */
static v3 xy_to_xyz(v2 a)
{
    v3 r = { a.x / a.y, 1.0f, (1.0f - a.x - a.y) / a.y };
    return r;
}
/* const_algebra.rs:69-71 */
static float dot3(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
/* const_algebra.rs:73-79 */
static v3 cross3(v3 a, v3 b)
{
    v3 r = { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x };
    return r;
}

/* constants_from_primaries, lib.rs:203-218: returns (kr, kb). */
static v2 constants_from_primaries(v2 r, v2 g, v2 b, v2 w)
{
    v3 r_xyz = xy_to_xyz(r), g_xyz = xy_to_xyz(g), b_xyz = xy_to_xyz(b), w_xyz = xy_to_xyz(w);
    v3 x_rgb = { r_xyz.x, g_xyz.x, b_xyz.x };
    v3 y_rgb = { r_xyz.y, g_xyz.y, b_xyz.y };
    v3 z_rgb = { r_xyz.z, g_xyz.z, b_xyz.z };
    float mul = 1.0f / dot3(x_rgb, cross3(y_rgb, z_rgb));
    v2 k = { dot3(w_xyz, cross3(g_xyz, b_xyz)) * mul, dot3(w_xyz, cross3(r_xyz, g_xyz)) * mul };
    return k;
}

/* matrix ids: 0 = BT709, 1 = BT601_525, 2 = BT601_625 (constants.rs:3-18). */
static v2 matrix_constants(int matrix)
{
    const v2 d65 = { 0.3127f, 0.3290f };
    v2 r, g, b;
    switch (matrix) {
    default:
    case 0: r = (v2){ 0.640f, 0.330f }; g = (v2){ 0.300f, 0.600f }; b = (v2){ 0.150f, 0.060f }; break;
    case 1: r = (v2){ 0.630f, 0.340f }; g = (v2){ 0.310f, 0.595f }; b = (v2){ 0.155f, 0.070f }; break;
    case 2: r = (v2){ 0.640f, 0.330f }; g = (v2){ 0.290f, 0.600f }; b = (v2){ 0.150f, 0.060f }; break;
    }
    return constants_from_primaries(r, g, b, d65);
}

/* ColorRange impls, lib.rs:77-169.  full_range != 0 is `Full` (the reference host code
 * todo!()s it, cuda-colorspace/src/lib.rs:45-52, but the kernel template supports it). */
typedef struct { uint32_t min, neutral, luma_range, chroma_range; } range_t;
static range_t color_range(int bits, int full_range)
{
    range_t r;
    r.neutral = 1u << (bits - 1);
    if (full_range) {
        r.min = 0;
        r.luma_range = (1u << bits) - 1;
        r.chroma_range = (1u << bits) - 1;
    } else {
        r.min = 16u << (bits - 8);
        r.luma_range = (235u << (bits - 8)) - r.min;
        r.chroma_range = (240u << (bits - 8)) - r.min;
    }
    return r;
}

/* MatrixCoefficients::coefficients, lib.rs:183-201: out = {y, r, b, g1, g2}. */
void oracle_yuv_coefficients(int matrix, int bits, int full_range, float out[5])
{
    v2 k = matrix_constants(matrix);
    float kr = k.x, kb = k.y;
    range_t cr = color_range(bits, full_range);
    float y_coeff = 1.0f / (float)cr.luma_range;
    float r_coeff = 2.0f * (1.0f - kr) * 1.0f / (float)cr.chroma_range;
    float b_coeff = 2.0f * (1.0f - kb) * 1.0f / (float)cr.chroma_range;
    float kg = 1.0f - kr - kb;
    float g_coeff1 = -2.0f * (1.0f - kb) * kb / kg * 1.0f / (float)cr.chroma_range;
    float g_coeff2 = -2.0f * (1.0f - kr) * kr / kg * 1.0f / (float)cr.chroma_range;
    out[0] = y_coeff; out[1] = r_coeff; out[2] = b_coeff; out[3] = g_coeff1; out[4] = g_coeff2;
}

void oracle_matrix_kr_kb(int matrix, float out[2])
{
    v2 k = matrix_constants(matrix);
    out[0] = k.x; out[1] = k.y;
}

/* BT709::eotf, lib.rs:220-236 (identical for the BT601 variants :247-281); powf_fast -> powf. */
static float bt709_eotf(float value)
{
    const float BETA = 0.018053968510807f;
    const float ALPHA = 1.0f + 5.5f * BETA;
    const float THRESHOLD = 0.08124285829863521110029445797874f;
    if (value >= THRESHOLD)
        return powf((value + (ALPHA - 1.0f)) / ALPHA, 1.0f / 0.45f);
    return value / 4.5f;
}

static float clamp01(float v)
{
    /* f32::max / f32::min semantics (NaN-ignoring), biplanar.rs:65-67 */
    v = fmaxf(v, 0.0f);
    return fminf(v, 1.0f);
}

/* One body for both sample widths.  bits = 8 (NV12, u8) or 16 (P016, u16 MSB-aligned).
 * y_plane / uv_plane are device-layout pointers with a shared pitch in bytes
 * (cudarse-video/src/dec.rs:299-366: UV = Y + pitch * coded_height). */
static void yuv420_to_linear(const void *y_plane, const void *uv_plane, size_t pitch, int bits,
                             int matrix, int full_range, int w, int h, float *out)
{
    float co[5];
    oracle_yuv_coefficients(matrix, bits, full_range, co);
    const float y_coeff = co[0], r_coeff = co[1], b_coeff = co[2], g_coeff1 = co[3], g_coeff2 = co[4];
    range_t cr = color_range(bits, full_range);
    size_t n = (size_t)w * h;
    /* the kernel runs one thread per 2x2 quad over (width/2, height/2): kernel.rs:53-79 */
    for (int qy = 0; qy < (h + 1) / 2; qy++) {
        for (int qx = 0; qx < (w + 1) / 2; qx++) {
            uint32_t u, v;
            if (bits == 8) {
                const uint8_t *p = (const uint8_t *)uv_plane + qy * pitch + 2 * qx;
                u = p[0]; v = p[1];
            } else {
                const uint16_t *p = (const uint16_t *)((const uint8_t *)uv_plane + qy * pitch) + 2 * qx;
                u = p[0]; v = p[1];
            }
            float cb = (float)((int32_t)u - (int32_t)cr.neutral);
            float crv = (float)((int32_t)v - (int32_t)cr.neutral);
            float r_ = r_coeff * crv;
            float g_ = fmaf(g_coeff1, cb, g_coeff2 * crv);
            float b_ = b_coeff * cb;
            for (int iy = 0; iy <= 1; iy++) {
                int y = 2 * qy + iy;
                if (y >= h) continue;
                for (int ix = 0; ix <= 1; ix++) {
                    int x = 2 * qx + ix;
                    if (x >= w) continue;
                    uint32_t s;
                    if (bits == 8)
                        s = ((const uint8_t *)y_plane + y * pitch)[x];
                    else
                        s = ((const uint16_t *)((const uint8_t *)y_plane + y * pitch))[x];
                    if (s < cr.min) s = cr.min;
                    float luma = (float)(s - cr.min) * y_coeff;
                    float r = luma + r_;
                    float g = luma + g_;
                    float b = luma + b_;
                    size_t o = (size_t)y * w + x;
                    out[o] = clamp01(bt709_eotf(r));
                    out[n + o] = clamp01(bt709_eotf(g));
                    out[2 * n + o] = clamp01(bt709_eotf(b));
                }
            }
        }
    }
}

void oracle_linear_from_nv12(const uint8_t *y_plane, const uint8_t *uv_plane, size_t pitch,
                             int matrix, int full_range, int w, int h, float *out)
{
    yuv420_to_linear(y_plane, uv_plane, pitch, 8, matrix, full_range, w, h, out);
}

void oracle_linear_from_p016(const uint16_t *y_plane, const uint16_t *uv_plane, size_t pitch,
                             int matrix, int full_range, int w, int h, float *out)
{
    yuv420_to_linear(y_plane, uv_plane, pitch, 16, matrix, full_range, w, h, out);
}

/* ------------------------------------------------------------------------------------ */
/* downscale_by_2, cpu.rs:545-579.                                                       */
/* ------------------------------------------------------------------------------------ */
void oracle_downscale_by_2(const float *in, int in_w, int in_h, float *out)
{
    int out_w = (in_w + 1) / 2, out_h = (in_h + 1) / 2;
    size_t n_in = (size_t)in_w * in_h, n_out = (size_t)out_w * out_h;
    const float normalize = 1.0f / 4.0f;
    for (int c = 0; c < 3; c++)
        for (int oy = 0; oy < out_h; oy++)
            for (int ox = 0; ox < out_w; ox++) {
                float sum = 0.0f;
                for (int iy = 0; iy < 2; iy++)
                    for (int ix = 0; ix < 2; ix++) {
                        int x = ox * 2 + ix; if (x > in_w - 1) x = in_w - 1;
                        int y = oy * 2 + iy; if (y > in_h - 1) y = in_h - 1;
                        sum += in[c * n_in + (size_t)y * in_w + x];
                    }
                out[c * n_out + (size_t)oy * out_w + ox] = sum * normalize;
            }
}

/* ------------------------------------------------------------------------------------ */
/* linear RGB -> XYB (rescaled positive).  cpu.rs:421-496.                               */
/* ------------------------------------------------------------------------------------ */
void oracle_opsin_constants(float out[12])
{
    const float K_M02 = 0.078f, K_M00 = 0.30f, K_M01 = 1.0f - K_M02 - K_M00;
    const float K_M12 = 0.078f, K_M10 = 0.23f, K_M11 = 1.0f - K_M12 - K_M10;
    const float K_M20 = 0.24342269f, K_M21 = 0.20476745f, K_M22 = 1.0f - K_M20 - K_M21;
    const float K_B0 = 0.0037930734f;
    const float K_B0_ROOT = 0.1559542025327239180319220163705f;
    float m[12] = { K_M00, K_M01, K_M02, K_M10, K_M11, K_M12, K_M20, K_M21, K_M22, K_B0, K_B0_ROOT, 0 };
    memcpy(out, m, sizeof(m));
}

static void px_linear_rgb_to_xyb(const float m[12], float r, float g, float b, float *ox, float *oy,
                                 float *ob)
{
    /* opsin_absorbance, cpu.rs:471-496 */
    float rg = fmaf(m[0], r, fmaf(m[1], g, fmaf(m[2], b, m[9])));
    float gr = fmaf(m[3], r, fmaf(m[4], g, fmaf(m[5], b, m[9])));
    float bb = fmaf(m[6], r, fmaf(m[7], g, fmaf(m[8], b, m[9])));
    /* cpu.rs:460-469 */
    rg = cbrtf(fmaxf(rg, 0.0f)) - m[10];
    gr = cbrtf(fmaxf(gr, 0.0f)) - m[10];
    bb = cbrtf(fmaxf(bb, 0.0f)) - m[10];
    float x = 0.5f * (rg - gr);
    float y = 0.5f * (rg + gr);
    *ox = fmaf(x, 14.0f, 0.42f);
    *oy = y + 0.01f;
    *ob = bb - y + 0.55f;
}

void oracle_linear_to_xyb(const float *lin, int w, int h, float *xyb)
{
    float m[12];
    oracle_opsin_constants(m);
    size_t n = (size_t)w * h;
    for (size_t i = 0; i < n; i++)
        px_linear_rgb_to_xyb(m, lin[i], lin[n + i], lin[2 * n + i], &xyb[i], &xyb[n + i], &xyb[2 * n + i]);
}

/* ------------------------------------------------------------------------------------ */
/* Recursive Gaussian, sigma = 1.5 (Charalampidis 2016).  cpu.rs:921-1115.               */
/* ------------------------------------------------------------------------------------ */
#define RG_RADIUS 5
static const float VERT_MUL_IN_1 = 0.055295236f, VERT_MUL_IN_3 = -0.058836687f, VERT_MUL_IN_5 = 0.012955819f;
static const float VERT_MUL_PREV_1 = -1.9021131f, VERT_MUL_PREV_3 = -1.1755705f,
                   VERT_MUL_PREV_5 = -0.00000000000000012246469f;
static const float MUL_IN_1 = 0.055295236f, MUL_IN_3 = -0.058836687f, MUL_IN_5 = 0.012955819f;
static const float MUL_PREV_1 = 1.9021131f, MUL_PREV_3 = 1.1755705f, MUL_PREV_5 = 0.00000000000000012246469f;
static const float MUL_PREV2_1 = -1.0f, MUL_PREV2_3 = -1.0f, MUL_PREV2_5 = -1.0f;

void oracle_rg_constants(float out[9])
{
    out[0] = MUL_IN_1; out[1] = MUL_IN_3; out[2] = MUL_IN_5;
    out[3] = MUL_PREV_1; out[4] = MUL_PREV_3; out[5] = MUL_PREV_5;
    out[6] = MUL_PREV2_1; out[7] = MUL_PREV2_3; out[8] = MUL_PREV2_5;
}

/* horizontal_row, cpu.rs:967-1022 */
static void horizontal_row(const float *input, float *output, int width)
{
    const int big_n = RG_RADIUS;
    float prev_1 = 0, prev_3 = 0, prev_5 = 0, prev2_1 = 0, prev2_3 = 0, prev2_5 = 0;
    for (int n = -big_n + 1; n < width; n++) {
        int left = n - big_n - 1, right = n + big_n - 1;
        float left_val = left >= 0 ? input[left] : 0.0f;
        float right_val = right < width ? input[right] : 0.0f;
        float sum = left_val + right_val;

        float out_1 = sum * MUL_IN_1;
        float out_3 = sum * MUL_IN_3;
        float out_5 = sum * MUL_IN_5;

        out_1 = fmaf(MUL_PREV2_1, prev2_1, out_1);
        out_3 = fmaf(MUL_PREV2_3, prev2_3, out_3);
        out_5 = fmaf(MUL_PREV2_5, prev2_5, out_5);
        prev2_1 = prev_1; prev2_3 = prev_3; prev2_5 = prev_5;

        out_1 = fmaf(MUL_PREV_1, prev_1, out_1);
        out_3 = fmaf(MUL_PREV_3, prev_3, out_3);
        out_5 = fmaf(MUL_PREV_5, prev_5, out_5);
        prev_1 = out_1; prev_3 = out_3; prev_5 = out_5;

        if (n >= 0)
            output[n] = out_1 + out_3 + out_5;
    }
}

/* horizontal_pass, cpu.rs:955-965 */
void oracle_blur_horizontal(const float *in, float *out, int w, int h)
{
    for (int y = 0; y < h; y++)
        horizontal_row(in + (size_t)y * w, out + (size_t)y * w, w);
}

/* vertical_pass, cpu.rs:1054-1115.  The reference processes columns in chunks of
 * 128 / 32 / 1 (vertical_pass_chunked :1024-1051); columns are independent, so the chunking
 * changes no arithmetic and one column at a time is restated here. */
void oracle_blur_vertical(const float *in, float *out, int w, int h)
{
    const int big_n = RG_RADIUS;
    for (int x = 0; x < w; x++) {
        float prev_1 = 0, prev_3 = 0, prev_5 = 0, prev2_1 = 0, prev2_3 = 0, prev2_5 = 0;
        for (int n = -big_n + 1; n < h; n++) {
            int top = n - big_n - 1, bottom = n + big_n - 1;
            float top_v = top >= 0 ? in[(size_t)top * w + x] : 0.0f;
            float bot_v = bottom < h ? in[(size_t)bottom * w + x] : 0.0f;
            float sum = top_v + bot_v;

            float o1 = fmaf(prev_1, VERT_MUL_PREV_1, prev2_1);
            float o3 = fmaf(prev_3, VERT_MUL_PREV_3, prev2_3);
            float o5 = fmaf(prev_5, VERT_MUL_PREV_5, prev2_5);
            o1 = fmaf(sum, VERT_MUL_IN_1, -o1);
            o3 = fmaf(sum, VERT_MUL_IN_3, -o3);
            o5 = fmaf(sum, VERT_MUL_IN_5, -o5);

            if (n >= 0)
                out[(size_t)n * w + x] = o1 + o3 + o5;

            prev2_1 = prev_1; prev2_3 = prev_3; prev2_5 = prev_5;
            prev_1 = o1; prev_3 = o3; prev_5 = o5;
        }
    }
}

/* Blur::blur_plane, cpu.rs:921-928: horizontal into temp, then vertical. */
void oracle_blur_plane(const float *in, float *out, float *temp, int w, int h)
{
    oracle_blur_horizontal(in, temp, w, h);
    oracle_blur_vertical(temp, out, w, h);
}

/* ------------------------------------------------------------------------------------ */
/* Error maps and their norms.  cpu.rs:581-683.                                          */
/* ------------------------------------------------------------------------------------ */
/* The f32 part of both maps at one pixel: the SSIM' quotient num_m * num_s / denom_s (cpu.rs:604-627) and the edge
 * map's a = |x2 - mu2|, b = |x1 - mu1| (cpu.rs:658-662).  Everything after these three values is f64 in the reference. */
static inline float ssim_quotient(float mu1, float mu2, float s11, float s22, float s12)
{
    const float C2 = 0.0009f;
    float mu11 = mu1 * mu1, mu22 = mu2 * mu2, mu12 = mu1 * mu2;
    float mu_diff = mu1 - mu2;
    float num_m = fmaf(mu_diff, -mu_diff, 1.0f);
    float num_s = fmaf(2.0f, s12 - mu12, C2);
    float denom_s = (s11 - mu11) + (s22 - mu22) + C2;
    return (num_m * num_s) / denom_s;
}

static inline void edge_inputs(float x1, float mu1, float x2, float mu2, float *a, float *b)
{
    *a = fabsf(x2 - mu2);
    *b = fabsf(x1 - mu1);
}

/* ssim_map: out6 = {L1,L4} x 3 channels as plane_averages[c*2 + n] */
static void ssim_map(int w, int h, const float *m1, const float *m2, const float *s11,
                     const float *s22, const float *s12, double out6[6])
{
    size_t n = (size_t)w * h;
    double one_per_pixels = 1.0 / (double)n;
    for (int c = 0; c < 3; c++) {
        double sum0 = 0.0, sum1 = 0.0;
        for (size_t i = 0; i < n; i++) {
            size_t k = c * n + i;
            double d = 1.0 - (double)ssim_quotient(m1[k], m2[k], s11[k], s22[k], s12[k]);
            d = d > 0.0 ? d : 0.0; /* f64::max(0.0); NaN -> 0.0 like Rust's max */
            if (d != d) d = 0.0;
            sum0 += d;
            double d2 = d * d; /* powi(4) */
            sum1 += d2 * d2;
        }
        out6[c * 2] = one_per_pixels * sum0;
        out6[c * 2 + 1] = sqrt(sqrt(one_per_pixels * sum1));
    }
}

/* edge_diff_map: out12 = plane_averages[c*4 + {art L1, art L4, det L1, det L4}] */
static void edge_diff_map(int w, int h, const float *img1, const float *mu1, const float *img2,
                          const float *mu2, double out12[12])
{
    size_t n = (size_t)w * h;
    double one_per_pixels = 1.0 / (double)n;
    for (int c = 0; c < 3; c++) {
        double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
        for (size_t i = 0; i < n; i++) {
            size_t k = c * n + i;
            float a, b;
            edge_inputs(img1[k], mu1[k], img2[k], mu2[k], &a, &b);
            double d1 = (1.0 + (double)a) / (1.0 + (double)b) - 1.0;
            double artifact = d1 > 0.0 ? d1 : 0.0;
            s0 += artifact;
            double a2 = artifact * artifact;
            s1 += a2 * a2;
            double detail_lost = -d1 > 0.0 ? -d1 : 0.0;
            s2 += detail_lost;
            double l2 = detail_lost * detail_lost;
            s3 += l2 * l2;
        }
        out12[c * 4] = one_per_pixels * s0;
        out12[c * 4 + 1] = sqrt(sqrt(one_per_pixels * s1));
        out12[c * 4 + 2] = one_per_pixels * s2;
        out12[c * 4 + 3] = sqrt(sqrt(one_per_pixels * s3));
    }
}

/* WEIGHT, cpu.rs:729-838 (identical to ssimulacra2-cuda/src/lib.rs:454-584): tuned model
 * parameters of SSIMULACRA 2.1, order [channel][scale][norm L1,L4][ssim, artifact, detail]. */
static const double WEIGHT[108] = {
    0.0, 0.0007376606707406586, 0.0, 0.0, 0.0007793481682867309, 0.0,
    0.0, 0.0004371155730107379, 0.0, 1.1041726426657346, 0.00066284834129271, 0.00015231632783718752,
    0.0, 0.0016406437456599754, 0.0, 1.8422455520539298, 11.441172603757666, 0.0,
    0.0007989109436015163, 0.000176816438078653, 0.0, 1.8787594979546387, 10.94906990605142, 0.0,
    0.0007289346991508072, 0.9677937080626833, 0.0, 0.00014003424285435884, 0.9981766977854967, 0.00031949755934435053,
    0.0004550992113792063, 0.0, 0.0, 0.0013648766163243398, 0.0, 0.0,
    0.0, 0.0, 0.0, 7.466890328078848, 0.0, 17.445833984131262,
    0.0006235601634041466, 0.0, 0.0, 6.683678146179332, 0.00037724407979611296, 1.027889937768264,
    225.20515300849274, 0.0, 0.0, 19.213238186143016, 0.0011401524586618361, 0.001237755635509985,
    176.39317598450694, 0.0, 0.0, 24.43300999870476, 0.28520802612117757, 0.0004485436923833408,
    0.0, 0.0, 0.0, 34.77906344483772, 44.835625328877896, 0.0,
    0.0, 0.0, 0.0, 0.0, 0.0, 0.0,
    0.0, 0.0008680556573291698, 0.0, 0.0, 0.0, 0.0,
    0.0, 0.0005313191874358747, 0.0, 0.00016533814161379112, 0.0, 0.0,
    0.0, 0.0, 0.0, 0.0004179171803251336, 0.0017290828234722833, 0.0,
    0.0020827005846636437, 0.0, 0.0, 8.826982764996862, 23.19243343998926, 0.0,
    95.1080498811086, 0.9863978034400682, 0.9834382792465353, 0.0012286405048278493, 171.2667255897307, 0.9807858872435379,
    0.0, 0.0, 0.0, 0.0005130064588990679, 0.0, 0.00010854057858411537,
};

void oracle_weights(double out[108]) { memcpy(out, WEIGHT, sizeof(WEIGHT)); }

/* Msssim::score, cpu.rs:728-871.  ssim6[s][c*2+n], edge12[s][c*4+n(+2)]. */
double oracle_score_from_averages(int nscales, const double (*ssim6)[6], const double (*edge12)[12])
{
    double ssim = 0.0;
    int i = 0;
    for (int c = 0; c < 3; c++)
        for (int s = 0; s < nscales; s++)
            for (int n = 0; n < 2; n++) {
                ssim = fma(WEIGHT[i], fabs(ssim6[s][c * 2 + n]), ssim); i++;
                ssim = fma(WEIGHT[i], fabs(edge12[s][c * 4 + n]), ssim); i++;
                ssim = fma(WEIGHT[i], fabs(edge12[s][c * 4 + n + 2]), ssim); i++;
            }
    ssim *= 0.9562382616834844;
    ssim = fma(6.248496625763138e-5 * ssim * ssim, ssim,
               fma(2.326765642916932, ssim, -0.020884521182843837 * ssim * ssim));
    if (ssim > 0.0)
        ssim = fma(pow(ssim, 0.6276336467831387), -10.0, 100.0);
    else
        ssim = 100.0;
    return ssim;
}

/* The per-scale stages of compute_frame_ssimulacra2 (cpu.rs:342-410): downscale, XYB, the five blurred planes. */
typedef struct {
    int w, h; /* size of the current scale */
    float *img1, *img2, *tmp, *x1, *x2, *mul, *temp, *s11, *s22, *s12, *mu1, *mu2;
} pyramid_t;

static void pyramid_init(pyramid_t *p, const float *ref_lin, const float *dis_lin, int w0, int h0)
{
    size_t n0 = (size_t)w0 * h0;
    p->w = w0; p->h = h0;
    p->img1 = malloc(3 * n0 * sizeof(float)); p->img2 = malloc(3 * n0 * sizeof(float));
    p->tmp = malloc(3 * n0 * sizeof(float));
    p->x1 = malloc(3 * n0 * sizeof(float)); p->x2 = malloc(3 * n0 * sizeof(float));
    p->mul = malloc(3 * n0 * sizeof(float)); p->temp = malloc(n0 * sizeof(float));
    p->s11 = malloc(3 * n0 * sizeof(float)); p->s22 = malloc(3 * n0 * sizeof(float));
    p->s12 = malloc(3 * n0 * sizeof(float)); p->mu1 = malloc(3 * n0 * sizeof(float));
    p->mu2 = malloc(3 * n0 * sizeof(float));
    memcpy(p->img1, ref_lin, 3 * n0 * sizeof(float));
    memcpy(p->img2, dis_lin, 3 * n0 * sizeof(float));
}

static void pyramid_free(pyramid_t *p)
{
    free(p->img1); free(p->img2); free(p->tmp); free(p->x1); free(p->x2); free(p->mul); free(p->temp);
    free(p->s11); free(p->s22); free(p->s12); free(p->mu1); free(p->mu2);
}

/* Move to scale `scale` (called for 0, 1, 2, ... in turn): the downscaled linear images.  Returns 0 when the image of
 * the previous scale is smaller than 8x8 (cpu.rs:359): that scale and every later one do not exist. */
static int pyramid_down(pyramid_t *p, int scale)
{
    int w = p->w, h = p->h;
    if (w < 8 || h < 8)
        return 0;
    if (scale > 0) {
        oracle_downscale_by_2(p->img1, w, h, p->tmp);
        int nw = (w + 1) / 2, nh = (h + 1) / 2;
        memcpy(p->img1, p->tmp, 3 * (size_t)nw * nh * sizeof(float));
        oracle_downscale_by_2(p->img2, w, h, p->tmp);
        memcpy(p->img2, p->tmp, 3 * (size_t)nw * nh * sizeof(float));
        p->w = nw; p->h = nh;
    }
    return 1;
}

/* XYB and the five blurred planes of the current scale. */
static void pyramid_planes(pyramid_t *p)
{
    int w = p->w, h = p->h;
    size_t n = (size_t)w * h;
    oracle_linear_to_xyb(p->img1, w, h, p->x1);
    oracle_linear_to_xyb(p->img2, w, h, p->x2);

    /* image_multiply + blur, cpu.rs:388-399 */
    for (size_t i = 0; i < 3 * n; i++) p->mul[i] = p->x1[i] * p->x1[i];
    for (int c = 0; c < 3; c++) oracle_blur_plane(p->mul + c * n, p->s11 + c * n, p->temp, w, h);
    for (size_t i = 0; i < 3 * n; i++) p->mul[i] = p->x2[i] * p->x2[i];
    for (int c = 0; c < 3; c++) oracle_blur_plane(p->mul + c * n, p->s22 + c * n, p->temp, w, h);
    for (size_t i = 0; i < 3 * n; i++) p->mul[i] = p->x1[i] * p->x2[i];
    for (int c = 0; c < 3; c++) oracle_blur_plane(p->mul + c * n, p->s12 + c * n, p->temp, w, h);
    for (int c = 0; c < 3; c++) oracle_blur_plane(p->x1 + c * n, p->mu1 + c * n, p->temp, w, h);
    for (int c = 0; c < 3; c++) oracle_blur_plane(p->x2 + c * n, p->mu2 + c * n, p->temp, w, h);
}

/* compute_frame_ssimulacra2, cpu.rs:342-410, on planar linear RGB inputs.
 * norms[108] (optional) receives the per-scale/per-channel averages in WEIGHT order for a
 * full 6-scale run: norms[c*36 + s*6 + n*3 + m], n in {L1,L4}, m in {ssim, artifact, detail};
 * entries of scales that were skipped (image < 8x8 at that scale, cpu.rs:359) are 0.
 * Returns the number of scales processed. */
int oracle_ssimu2_linear_planar(const float *ref_lin, const float *dis_lin, int w0, int h0,
                                double *score, double *norms)
{
    pyramid_t p;
    double ssim6[NUM_SCALES][6], edge12[NUM_SCALES][12];
    int nscales = 0;
    pyramid_init(&p, ref_lin, dis_lin, w0, h0);
    if (norms) memset(norms, 0, 108 * sizeof(double));

    for (int scale = 0; scale < NUM_SCALES; scale++) {
        if (!pyramid_down(&p, scale))
            break;
        pyramid_planes(&p);
        ssim_map(p.w, p.h, p.mu1, p.mu2, p.s11, p.s22, p.s12, ssim6[scale]);
        edge_diff_map(p.w, p.h, p.x1, p.mu1, p.x2, p.mu2, edge12[scale]);
        if (norms)
            for (int c = 0; c < 3; c++)
                for (int nn = 0; nn < 2; nn++) {
                    norms[c * 36 + scale * 6 + nn * 3 + 0] = ssim6[scale][c * 2 + nn];
                    norms[c * 36 + scale * 6 + nn * 3 + 1] = edge12[scale][c * 4 + nn];
                    norms[c * 36 + scale * 6 + nn * 3 + 2] = edge12[scale][c * 4 + nn + 2];
                }
        nscales++;
    }
    if (score)
        *score = oracle_score_from_averages(nscales, ssim6, edge12);
    pyramid_free(&p);
    return nscales;
}

/* The per-pixel inputs of the error maps of one scale, as ssim_map and edge_diff_map see them: q = the SSIM' quotient,
 * a = |x2 - mu2|, b = |x1 - mu1|, each float[3][h_s][w_s] for the w_s x h_s image of that scale.  From these the maps
 * are d = max(1 - q, 0) and d1 = (1 + a) / (1 + b) - 1 in f64.  Returns 0, or -1 when the scale does not exist. */
int oracle_map_inputs(const float *ref_lin, const float *dis_lin, int w0, int h0, int scale, float *q, float *a, float *b)
{
    pyramid_t p;
    int ok = scale >= 0 && scale < NUM_SCALES;
    pyramid_init(&p, ref_lin, dis_lin, w0, h0);
    for (int s = 0; ok && s <= scale; s++)
        ok = pyramid_down(&p, s);
    if (ok) {
        pyramid_planes(&p);
        size_t n = (size_t)p.w * p.h;
        for (size_t k = 0; k < 3 * n; k++) {
            q[k] = ssim_quotient(p.mu1[k], p.mu2[k], p.s11[k], p.s22[k], p.s12[k]);
            edge_inputs(p.x1[k], p.mu1[k], p.x2[k], p.mu2[k], &a[k], &b[k]);
        }
    }
    pyramid_free(&p);
    return ok ? 0 : -1;
}

/* Front-end + metric in one call, one per input format of the boundary
 * (turbo-metrics/src/lib.rs:125-130 HwFrame; color.rs:96-116). */
int oracle_ssimu2_srgb8(const uint8_t *ref, size_t ref_pitch, const uint8_t *dis, size_t dis_pitch,
                        int w, int h, double *score, double *norms)
{
    size_t n = (size_t)w * h;
    float *a = malloc(3 * n * sizeof(float)), *b = malloc(3 * n * sizeof(float));
    oracle_linear_from_srgb8(ref, ref_pitch, w, h, a);
    oracle_linear_from_srgb8(dis, dis_pitch, w, h, b);
    int r = oracle_ssimu2_linear_planar(a, b, w, h, score, norms);
    free(a); free(b);
    return r;
}

int oracle_ssimu2_yuv420(const void *ref_y, const void *ref_uv, size_t ref_pitch, const void *dis_y,
                         const void *dis_uv, size_t dis_pitch, int bits, int matrix, int full_range,
                         int w, int h, double *score, double *norms)
{
    size_t n = (size_t)w * h;
    float *a = malloc(3 * n * sizeof(float)), *b = malloc(3 * n * sizeof(float));
    yuv420_to_linear(ref_y, ref_uv, ref_pitch, bits, matrix, full_range, w, h, a);
    yuv420_to_linear(dis_y, dis_uv, dis_pitch, bits, matrix, full_range, w, h, b);
    int r = oracle_ssimu2_linear_planar(a, b, w, h, score, norms);
    free(a); free(b);
    return r;
}

int oracle_ssimu2_linearf32(const float *ref, size_t ref_pitch, const float *dis, size_t dis_pitch,
                            int w, int h, double *score, double *norms)
{
    size_t n = (size_t)w * h;
    float *a = malloc(3 * n * sizeof(float)), *b = malloc(3 * n * sizeof(float));
    oracle_linear_from_linearf32(ref, ref_pitch, w, h, a);
    oracle_linear_from_linearf32(dis, dis_pitch, w, h, b);
    int r = oracle_ssimu2_linear_planar(a, b, w, h, score, norms);
    free(a); free(b);
    return r;
}
