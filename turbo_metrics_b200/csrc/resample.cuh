// resample.cuh -- k_resample: upscales the distorted frames of a scaled handle (ssimu2_source.width / height) to the
// reference's size, in their own sample domain, before the distorted side's front-end reads them (sm_100a).
//
// Filter: separable bicubic Catmull-Rom (Keys, a = -0.5), centre-aligned, clamp-to-edge, per plane grid.  The per-axis tap
// tables (first tap index i - 1 and four f32 weights per output coordinate) are built on the host (ssimu2_api.cu); here the
// arithmetic is fixed, horizontal first:
//   row r:  a = w0 * s0;  a = fmaf(w1, s1, a);  a = fmaf(w2, s2, a);  a = fmaf(w3, s3, a)     (x weights, 4 source samples)
//   out:    the same chain over the 4 row results with the y weights.
// u8 / u16 results are rounded half to even and clamped to the sample range, f32 results are stored as they are.  The
// CPU reference of the tests (tests/native/resample_ref.c) evaluates exactly this; compile with -fmad=false.
#pragma once
#include "ssimu2_kernels.cuh"

namespace ssimu2 {

constexpr int kRsTileX = 32;                // output pixels (per channel) of a tile's row
constexpr int kRsTileY = 32;                // output rows of a tile
constexpr int kRsThreads = 256;
// Source rows a tile's vertical taps reach when the plane is upscaled (in <= out): at most kRsTileY + 4.
constexpr int kRsRows = kRsTileY + 4;

struct RsAxis {
    const float4* w;   // [out] the 4 tap weights of output coordinate x
    const int* j0;     // [out] its first tap index, i - 1 (may be -1; taps are clamped to [0, in - 1] when read)
};

struct RsPlane {
    int in_w, in_h, out_w, out_h;   // per channel
    int tiles_x, tile0;             // tiles of this plane along x, index of its first tile in the launch
    RsAxis x, y;
    long long dst_off;              // byte offset of the plane in a staged frame
};

struct RsArgs {
    RsPlane pl[3];        // Y (or packed RGB), chroma (CbCr interleaved, or Cb), Cr (4:4:4 only)
    int nplanes;
    int tiles;            // tiles of all planes of one frame
    uint8_t* dst;         // staged frames: [frame of the launch][dst_stride]
    long long dst_stride;
    uint32_t dst_pitch;   // bytes, a multiple of 256
};

// Sample type and interleaved channels per plane of the formats a distorted side can have.
template <int FMT>
struct RsFmt {
    static constexpr bool f32 = FMT == kSRGBF32 || FMT == kLINEARF32;
    static constexpr bool u16 = FmtIs<FMT>::u16 || FMT == kSRGB16;
    using T = typename std::conditional<f32, float, typename std::conditional<u16, uint16_t, uint8_t>::type>::type;
    static constexpr int luma_ch = FmtIs<FMT>::yuv ? 1 : 3;                               // packed RGB: 3 channels
    static constexpr int chroma_ch = (FmtIs<FMT>::yuv420 || FmtIs<FMT>::yuv422) ? 2 : 1;  // interleaved CbCr
    static constexpr float vmax = u16 ? 65535.f : 255.f;
};

template <typename T>
__device__ __forceinline__ T rs_store_value(float a, float vmax)
{
    if constexpr (std::is_same<T, float>::value) {
        return a;
    } else {
        return (T)fminf(fmaxf(rintf(a), 0.f), vmax);   // round half to even, then clamp
    }
}

// One output tile of one plane with NCH interleaved channels.
template <int FMT, int NCH>
__device__ __forceinline__ void resample_tile(const RsArgs& a, const RsPlane& P, const uint8_t* src, uint32_t pitch, int tt,
                                              uint8_t* dst, float (*hs)[kRsTileX * 3])
{
    using T = typename RsFmt<FMT>::T;
    const int X0 = (tt % P.tiles_x) * kRsTileX, Y0 = (tt / P.tiles_x) * kRsTileY;
    const int tw = min(kRsTileX, P.out_w - X0), th = min(kRsTileY, P.out_h - Y0);
    const int cols = tw * NCH;
    // the source rows the tile's vertical taps reach (monotonic in y: the first tap of the first row to the last of the last)
    const int r_lo = max(P.y.j0[Y0], 0);
    const int r_hi = min(P.y.j0[Y0 + th - 1] + 3, P.in_h - 1);
    const int nrows = min(r_hi - r_lo + 1, kRsRows);
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    // horizontal pass: every source row of the tile, every output column and channel, into shared memory
    for (int c = cx; c < cols; c += 32) {
        const int x = X0 + c / NCH, ch = c % NCH;
        const float4 w = P.x.w[x];
        const int j0 = P.x.j0[x];
        const int s0 = min(max(j0, 0), P.in_w - 1) * NCH + ch, s1 = min(max(j0 + 1, 0), P.in_w - 1) * NCH + ch;
        const int s2 = min(max(j0 + 2, 0), P.in_w - 1) * NCH + ch, s3 = min(max(j0 + 3, 0), P.in_w - 1) * NCH + ch;
        for (int r = ry; r < nrows; r += kRsThreads / 32) {
            const T* row = reinterpret_cast<const T*>(src + (size_t)(r_lo + r) * pitch);   // 64-bit row base
            float acc = w.x * (float)row[s0];
            acc = fmaf(w.y, (float)row[s1], acc);
            acc = fmaf(w.z, (float)row[s2], acc);
            acc = fmaf(w.w, (float)row[s3], acc);
            hs[r][c] = acc;
        }
    }
    __syncthreads();
    // vertical pass over the row results, stored in the staged frame
    for (int r = ry; r < th; r += kRsThreads / 32) {
        const int y = Y0 + r;
        const float4 w = P.y.w[y];
        const int j0 = P.y.j0[y];
        const int k0 = min(max(j0, 0), P.in_h - 1) - r_lo, k1 = min(max(j0 + 1, 0), P.in_h - 1) - r_lo;
        const int k2 = min(max(j0 + 2, 0), P.in_h - 1) - r_lo, k3 = min(max(j0 + 3, 0), P.in_h - 1) - r_lo;
        T* out = reinterpret_cast<T*>(dst + P.dst_off + (size_t)y * a.dst_pitch) + X0 * NCH;
        for (int c = cx; c < cols; c += 32) {
            float acc = w.x * hs[k0][c];
            acc = fmaf(w.y, hs[k1][c], acc);
            acc = fmaf(w.z, hs[k2][c], acc);
            acc = fmaf(w.w, hs[k3][c], acc);
            out[c] = rs_store_value<T>(acc, RsFmt<FMT>::vmax);
        }
    }
}

// grid (a.tiles, 1, n): block (t, 0, z) resamples tile t (planes in order) of the distorted frame of pair frame0 + z into
// staged frame z.  The caller's frame is only assumed aligned to one sample.
template <int FMT>
__global__ void __launch_bounds__(kRsThreads) k_resample(const __grid_constant__ RsArgs a, const FramePair* __restrict__ in, int frame0)
{
    __shared__ float hs[kRsRows][kRsTileX * 3];
    const FrameIn f = in[frame0 + blockIdx.z].dis;
    uint8_t* dst = a.dst + (size_t)blockIdx.z * a.dst_stride;
    const int t = blockIdx.x;
    if (a.nplanes > 1 && t >= a.pl[1].tile0) {
        if (a.nplanes > 2 && t >= a.pl[2].tile0) {
            // 4:4:4 Cr: plane[1] + (plane[1] - plane[0]), modulo 2^64 as the layout rule states it
            const uint8_t* cr = (const uint8_t*)((uintptr_t)f.p1 + ((uintptr_t)f.p1 - (uintptr_t)f.p0));
            resample_tile<FMT, 1>(a, a.pl[2], cr, f.pitch, t - a.pl[2].tile0, dst, hs);
        } else {
            resample_tile<FMT, RsFmt<FMT>::chroma_ch>(a, a.pl[1], f.p1, f.pitch, t - a.pl[1].tile0, dst, hs);
        }
    } else {
        resample_tile<FMT, RsFmt<FMT>::luma_ch>(a, a.pl[0], f.p0, f.pitch, t, dst, hs);
    }
}

}  // namespace ssimu2
