// frame_layout.h -- the layout rule every submitted frame must meet (include/ssimu2_b200.h, ssimu2_frame), stated once for
// the single-GPU entry points (ssimu2_api.cu) and the shard API (ssimu2_shard.cpp).
#pragma once

#include "../../include/ssimu2_b200.h"

// One frame of format `fmt` (a valid ssimu2_format) and size width x height.
//  - The pitch holds a row: width samples of luma (YUV; and 2 * ceil(width / 2) samples of interleaved chroma), or width
//    pixels (packed RGB).
//  - Every load the front-end issues is aligned to one sample (1 byte: NV12, sRGB8; 2: P016, sRGB16; 4: the f32 formats).
//    Device frames: the plane addresses and the pitch are multiples of it.  Host frames are copied to 256-aligned staging
//    memory, so there the pitch and plane[1] - plane[0] (after plane[0]) are.
//  - Host frames: `bytes`, the count copied from plane[0], reaches the end of the last luma row and, for YUV, of the last
//    chroma row; otherwise the front-end would read past the frame's staging slot.
inline bool frame_layout_ok(int fmt, uint32_t width, uint32_t height, const ssimu2_frame* f, bool host, size_t bytes)
{
    if (!f || !f->plane[0] || f->pitch == 0) return false;
    const bool yuv = fmt == SSIMU2_FMT_NV12 || fmt == SSIMU2_FMT_P016;
    if (yuv && !f->plane[1]) return false;
    static const uint32_t sample_bytes[] = {1, 2, 1, 2, 4, 4};
    static const uint32_t samples_per_px[] = {1, 1, 3, 3, 3, 3};   // YUV: luma samples
    const uint64_t s = sample_bytes[fmt];
    const uint64_t luma_row = (uint64_t)width * samples_per_px[fmt] * s;
    const uint64_t chroma_row = yuv ? (uint64_t)(width + 1) / 2 * 2 * s : 0;
    const uint64_t pitch = f->pitch;
    if (pitch < luma_row || pitch < chroma_row || pitch % s) return false;
    if (!host) return f->plane[0] % s == 0 && (!yuv || f->plane[1] % s == 0);
    if (luma_row + (uint64_t)(height - 1) * pitch > bytes) return false;
    if (!yuv) return true;
    if (f->plane[1] <= f->plane[0]) return false;
    const uint64_t off = f->plane[1] - f->plane[0];
    return off % s == 0 && off < bytes && off + (uint64_t)((height + 1) / 2 - 1) * pitch + chroma_row <= bytes;
}
