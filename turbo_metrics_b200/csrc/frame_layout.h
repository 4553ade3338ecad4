// frame_layout.h -- the layout rule every submitted frame must meet (include/ssimu2_b200.h, ssimu2_frame), stated once for
// the single-GPU entry points (ssimu2_api.cu) and the shard API (ssimu2_shard.cpp).
#pragma once

#include "../../include/ssimu2_b200.h"

// Whether `fmt` is an ssimu2_format value (6 and 7 are not).
inline bool format_known(int fmt) { return (fmt >= SSIMU2_FMT_NV12 && fmt <= SSIMU2_FMT_LINEARF32) || (fmt >= SSIMU2_FMT_NV16 && fmt <= SSIMU2_FMT_YUV444P16); }
inline bool format_is_yuv(int fmt)
{
    return fmt == SSIMU2_FMT_NV12 || fmt == SSIMU2_FMT_P016 || (fmt >= SSIMU2_FMT_NV16 && fmt <= SSIMU2_FMT_YUV444P16);
}
// the formats SSIMU2_FLAG_P016_DEEP applies to: YUV with 16-bit samples
inline bool format_is_yuv16(int fmt) { return fmt == SSIMU2_FMT_P016 || fmt == SSIMU2_FMT_P216 || fmt == SSIMU2_FMT_YUV444P16; }

// One frame of format `fmt` (a valid ssimu2_format) and size width x height.
//  - The pitch holds a row: width samples of luma (YUV; and 2 * ceil(width / 2) samples of interleaved chroma for 4:2:0 and
//    4:2:2, width samples of Cb and of Cr for 4:4:4), or width pixels (packed RGB).
//  - Every load the front-end issues is aligned to one sample (1 byte: NV12, NV16, YUV444, sRGB8; 2: P016, P216, YUV444P16,
//    sRGB16; 4: the f32 formats).  Device frames: the plane addresses (4:4:4: and the Cr plane's, plane[1] + (plane[1] -
//    plane[0]), which must not wrap) and the pitch are multiples of it.  Host frames are copied to 256-aligned staging memory,
//    so there the pitch and plane[1] - plane[0] (after plane[0]) are.
//  - Host frames: `bytes`, the count copied from plane[0], reaches the end of the last luma row and, for YUV, of the last
//    chroma row (4:2:0: ceil(height / 2) rows; 4:2:2: height rows; 4:4:4: height rows of Cb, then of Cr); otherwise the
//    front-end would read past the frame's staging slot.
inline bool frame_layout_ok(int fmt, uint32_t width, uint32_t height, const ssimu2_frame* f, bool host, size_t bytes)
{
    if (!f || !f->plane[0] || f->pitch == 0) return false;
    const bool yuv = format_is_yuv(fmt);
    const bool yuv444 = fmt == SSIMU2_FMT_YUV444 || fmt == SSIMU2_FMT_YUV444P16;
    const bool yuv420 = fmt == SSIMU2_FMT_NV12 || fmt == SSIMU2_FMT_P016;
    if (yuv && !f->plane[1]) return false;
    // indexed by format: NV12 P016 SRGB8 SRGB16 SRGBF32 LINEARF32 - - NV16 P216 YUV444 YUV444P16
    static const uint32_t sample_bytes[] = {1, 2, 1, 2, 4, 4, 0, 0, 1, 2, 1, 2};
    static const uint32_t samples_per_px[] = {1, 1, 3, 3, 3, 3, 0, 0, 1, 1, 1, 1};   // YUV: luma samples
    const uint64_t s = sample_bytes[fmt];
    const uint64_t luma_row = (uint64_t)width * samples_per_px[fmt] * s;
    const uint64_t chroma_row = !yuv ? 0 : yuv444 ? luma_row : (uint64_t)(width + 1) / 2 * 2 * s;
    const uint64_t chroma_rows = yuv420 ? (height + 1) / 2 : height;
    const uint64_t pitch = f->pitch;
    if (pitch < luma_row || pitch < chroma_row || pitch % s) return false;
    if (!host) {
        if (f->plane[0] % s || (yuv && f->plane[1] % s)) return false;
        if (!yuv444) return true;
        // Cr = plane[1] + (plane[1] - plane[0]) (mod 2^64): aligned when both planes are; it must not wrap around either end
        const uint64_t p0 = f->plane[0], p1 = f->plane[1];
        return p1 >= p0 ? p1 - p0 <= UINT64_MAX - p1 : p0 - p1 <= p1;
    }
    if (luma_row + (uint64_t)(height - 1) * pitch > bytes) return false;
    if (!yuv) return true;
    if (f->plane[1] <= f->plane[0]) return false;
    const uint64_t off = f->plane[1] - f->plane[0];
    if (off % s || off >= bytes) return false;
    // the last chroma row (4:4:4: of the Cr plane, `off` past the Cb plane)
    const uint64_t cr = yuv444 ? off : 0;
    if (cr > bytes) return false;
    return off + cr + (chroma_rows - 1) * pitch + chroma_row <= bytes;
}
