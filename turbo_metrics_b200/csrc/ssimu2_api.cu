// ssimu2_api.cu -- host side of libssimu2_b200.so: the C ABI declared in include/ssimu2_b200.h.
//
// Mirrors the reference's metric op (crates/ssimulacra2-cuda/src/lib.rs:27-291) and the per-pair
// driver that calls it (crates/turbo-metrics/src/lib.rs:268-360), re-designed for throughput:
//   * a handle owns `ring` batch slots; each slot has its own stream, workspace and result buffers;
//   * pairs are collected into batches of `batch` and every batch is 3 kernel launches that cover
//     all frames and all 6 scales (the reference records a 305-node graph per pair and syncs the
//     host after every pair, lib.rs:342-352);
//   * the front-end (the only kernel that reads the caller's frames) can run per input group of a few pairs
//     (cfg.input_group), so that decoder surfaces are consumed soon after submit;
//   * only the f64 scores (and, for parity tests, the 108 norms) travel back to the host.
// There is no CPU fallback: without a usable CUDA device every call fails.
#include "../../include/ssimu2_b200.h"
#include "../../include/ssimu2_b200_debug.h"
#include "frame_layout.h"
#include "ssimu2_kernels.cuh"
#include "resample.cuh"

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

using namespace ssimu2;

namespace {

constexpr uint64_t kResultCap = 16384;  // tickets kept in the host/device result rings
constexpr uint32_t kDefaultBatch = 8;
constexpr uint32_t kDefaultRing = 3;

#define CU_TRY(expr)                                 \
    do {                                             \
        cudaError_t _e = (expr);                     \
        if (_e != cudaSuccess) return (int)_e;       \
    } while (0)

// Every entry point runs on the handle's device and leaves the caller's current device as it found it.
struct DeviceGuard {
    int prev = -1, dev;
    explicit DeviceGuard(int d) : dev(d)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; }
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard()
    {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
};

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_in = nullptr;      // dependency on the submitter's stream, recorded at submit time
    cudaEvent_t ev_done = nullptr;    // batch complete (results on host)
    cudaEvent_t ev_k[5] = {};         // per-kernel timing marks
    std::vector<cudaEvent_t> ev_fe;   // one per front-end launch of the current batch: "inputs consumed"
    std::vector<uint16_t> fe_seq;     // [batch] front-end launch that served pair i
    uint32_t fe_launches = 0;         // front-end launches of the current batch so far
    uint32_t fe_pairs = 0;            // pairs of the current batch whose front-end has been launched
    float* xyb = nullptr;             // [batch] XYB planes of all scales
    float* hb = nullptr;              // [batch] H-pass planes (split pipeline only)
    double* partials = nullptr;       // [batch][total_strips][18]
    double* norms_d = nullptr;        // [batch][108]
    double* scores_d = nullptr;       // [batch]
    double* norms_h = nullptr;        // pinned
    double* scores_h = nullptr;       // pinned
    double* tiles = nullptr;          // tile handle: k_hv<true>'s tile table [batch][tile_entries][18]
    double* tile_scores_d = nullptr;  // [batch][tiles_y][tiles_x]
    double* tile_scores_h = nullptr;  // pinned
    uint8_t* staging = nullptr;       // device staging for host frames: [batch][2][staging_frame_bytes]
    FramePair* in_h = nullptr;        // pinned frame table of the batch being recorded
    FramePair* in_d = nullptr;        // its device copy (uploaded per front-end launch)
    uint8_t* rs_frames = nullptr;     // scaled handle: the upscaled distorted frames of one front-end launch [rs_group][rs.dst_stride]
    FramePair* rs_in_h = nullptr;     // scaled handle: frame table of the distorted front-end (dis entries point at rs_frames)
    FramePair* rs_in_d = nullptr;     // its device copy
    TmaMaps maps{};                   // tensor maps of this slot's H-pass / XYB buffers, per scale (V pass)
    TmaMapsH maps_h{};                // (H pass)
    TmaMapsX maps_x{};                // (fused H+V kernel)
    f2* hstate = nullptr;             // k_hv hand-off records: [batch][total_recs][6][96]
    uint32_t* hvflags = nullptr;      // [batch][total_recs] + the work-item counter at the end
    uint32_t epoch = 0;               // launch counter of k_hv on this slot (flag value)
    uint32_t count = 0;               // pairs recorded
    uint64_t first_ticket = 0;
    bool inflight = false;            // fully launched, results not harvested yet
    bool timed = false, was_timed = false;
    void* dep_stream = nullptr;       // stream ev_in was last recorded on
    bool have_dep = false;
};

}  // namespace

struct ssimu2_handle {
    ssimu2_config cfg{};
    Geo geo{};                        // geometry + the reference side's coefficients and memo table
    // mixed sources (ssimu2_create_mixed with a distorted description that differs from cfg): the front-end runs once per
    // side, the distorted side with geo_dis (geo with that side's coefficients and memo table)
    bool mixed = false;
    int fmt[2] = {0, 0};              // ssimu2_format of the reference / distorted frames
    int fe_fmt[2] = {0, 0};           // their front-end formats (kP016A / kP216A / kYUV444P16A: with SSIMU2_FLAG_P016_DEEP)
    Geo geo_dis{};
    float* eotf_lut_dis = nullptr;
    uint32_t side_w[2] = {0, 0}, side_h[2] = {0, 0};   // size of the reference / distorted frames
    // scaled distorted frames (ssimu2_source.width / height smaller than the reference): k_resample upscales them into
    // rs_frames before the distorted side's front-end; rs holds the plane grids and tap tables (rs_tab), rs_group is the
    // most pairs one front-end launch covers
    bool scaled = false;
    RsArgs rs{};
    void* rs_tab = nullptr;
    uint32_t rs_group = 0;
    uint32_t batch = 0, ring = 0, input_group = 0;
    std::vector<Slot> slots;
    uint32_t cur = 0;
    int pipeline = 0;                 // 0 = fused (front-end, k_hv, finalize) / 1 = split (front-end, k_hpass, k_vpass, finalize)
    bool score_only = false;
    uint64_t next_ticket = 0;
    double* scores_ring_d = nullptr;  // [kResultCap] device score stream
    float* eotf_lut = nullptr;        // exact R / B transfer memo for YUV sources (see Geo)
    std::vector<double> res_scores;   // host result ring
    std::vector<double> res_norms;    // [kResultCap][108]
    std::vector<int32_t> res_slot;    // slot that served the ticket (for debug_read)
    size_t device_bytes = 0;
    size_t staging_frame_bytes = 0;
    uint64_t launches = 0;
    float last_ms[4] = {0, 0, 0, 0};
    double total_ms[4] = {0, 0, 0, 0};  // per-kernel device time summed over harvested batches
    uint64_t timed_batches = 0, timed_pairs = 0;
    uint64_t alg_bytes = 0, io_bytes = 0;
    unsigned char lite[kMaxScales] = {};   // score-only: channels without SSIM' per scale (HvArgs::lite)
    // tile scores (ssimu2_config.tile != 0): grid, entries of a frame's tile table, and the host ring of the last tile_cap maps
    uint32_t tile = 0, tiles_x = 0, tiles_y = 0;
    int tile_log2 = 0;
    size_t tile_entries = 0;
    uint64_t tile_cap = 0;
    std::vector<double> res_tiles;    // [tile_cap][tiles_y * tiles_x]
};

namespace {

// ---- colour coefficients (host, f32 arithmetic as in cuda-colorspace-kernel/src/lib.rs:183-218) ----
struct V3 { float x, y, z; };
static V3 xyz_of(float x, float y) { return V3{x / y, 1.0f, (1.0f - x - y) / y}; }
static float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static V3 cross(V3 a, V3 b) { return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

static void luma_constants(int matrix, float& kr, float& kb)
{
    // primaries: constants.rs:3-18
    float p[3][6] = {{0.640f, 0.330f, 0.300f, 0.600f, 0.150f, 0.060f},
                     {0.630f, 0.340f, 0.310f, 0.595f, 0.155f, 0.070f},
                     {0.640f, 0.330f, 0.290f, 0.600f, 0.150f, 0.060f}};
    const float* m = p[matrix];
    V3 r = xyz_of(m[0], m[1]), g = xyz_of(m[2], m[3]), b = xyz_of(m[4], m[5]), w = xyz_of(0.3127f, 0.3290f);
    V3 xr{r.x, g.x, b.x}, yr{r.y, g.y, b.y}, zr{r.z, g.z, b.z};
    float mul = 1.0f / dot(xr, cross(yr, zr));
    kr = dot(w, cross(g, b)) * mul;
    kb = dot(w, cross(r, g)) * mul;
}

static YuvCoef make_coef(int fmt, int matrix, int full_range)
{
    YuvCoef c{};
    if (!format_is_yuv(fmt)) return c;
    int bits = format_is_yuv16(fmt) ? 16 : 8;
    float kr, kb;
    luma_constants(matrix, kr, kb);
    uint32_t lmin, lrange, crange;
    if (full_range) {
        lmin = 0; lrange = (1u << bits) - 1; crange = (1u << bits) - 1;
    } else {
        lmin = 16u << (bits - 8);
        lrange = (235u << (bits - 8)) - lmin;
        crange = (240u << (bits - 8)) - lmin;
    }
    float kg = 1.0f - kr - kb;
    c.y = 1.0f / (float)lrange;
    c.r = 2.0f * (1.0f - kr) * 1.0f / (float)crange;
    c.b = 2.0f * (1.0f - kb) * 1.0f / (float)crange;
    c.g1 = -2.0f * (1.0f - kb) * kb / kg * 1.0f / (float)crange;
    c.g2 = -2.0f * (1.0f - kr) * kr / kg * 1.0f / (float)crange;
    c.luma_min = (int)lmin;
    c.neutral = 1 << (bits - 1);
    return c;
}

// the front-end format of a 16-bit YUV side with SSIMU2_FLAG_P016_DEEP
static int deep_fe_fmt(int fmt) { return fmt == kP016 ? kP016A : fmt == kP216 ? kP216A : kYUV444P16A; }

static int in_bytes_per_px(int fmt)
{
    switch (fmt) {
    case kNV12: return 3;       // 1.5 B x 2 images
    case kP016: return 6;
    case kNV16: return 4;       // 2 B x 2 images
    case kP216: return 8;
    case kYUV444: return 6;
    case kYUV444P16: return 12;
    case kSRGB8: return 6;
    case kSRGB16: return 12;
    default: return 24;
    }
}

static void build_geo(ssimu2_handle* h)
{
    Geo& g = h->geo;
    int w = (int)h->cfg.width, hh = (int)h->cfg.height;
    long long xyb_off = 0, hb_off = 0;
    int strips = 0, ns = 0, recs = 0;
    unsigned long long sum_px = 0, sum_px_ge1 = 0;
    for (int s = 0; s < kMaxScales; s++) {
        if (w < 8 || hh < 8) break;  // cpu.rs:359: tested on the size BEFORE this scale's downscale
        if (s > 0) { w = (w + 1) / 2; hh = (hh + 1) / 2; }
        ScaleDesc& d = g.sc[s];
        d.w = w; d.h = hh;
        d.pitch = (w + 31) / 32 * 32;
        d.n_bands = (hh + kHRows - 1) / kHRows;
        d.n_strips = (w + kVCols - 1) / kVCols;
        d.strip0 = strips;
        strips += d.n_strips;
        d.xyb_off = xyb_off;
        xyb_off += 6LL * hh * d.pitch;
        d.hb_off = hb_off;
        hb_off += 15LL * hh * d.pitch;
        d.nb = (hh + 4 + kXR - 1) / kXR;
        d.rec0 = recs;
        d.item0 = strips - d.n_strips;
        recs += d.n_strips * d.nb;
        sum_px += (unsigned long long)w * hh;
        if (s >= 1) sum_px_ge1 += (unsigned long long)w * hh;
        ns++;
    }
    g.nscales = ns;
    g.total_strips = strips;
    g.total_recs = recs;
    g.xyb_stride = xyb_off;
    g.hb_stride = hb_off;
    g.items_h = 0; g.items_v = 0;
    for (int s = 0; s < ns; s++) { g.items_h += g.sc[s].n_bands; g.items_v += g.sc[s].n_strips; }
    g.coef = make_coef(h->cfg.format, h->cfg.matrix, h->cfg.full_range);
    // SURVEY.md section 8(d): B_alg = 120*sum(P_s) + 2*in_0*P_0 + 72*sum_{s>=1}(P_s), in_0 = input bytes per pixel of the pair
    // (each side at its own bytes per pixel: in_bytes_per_px is per two images of one format)
    // (a scaled distorted side counts at its own size)
    const unsigned long long in2 = (unsigned long long)in_bytes_per_px(h->fmt[0]) * h->side_w[0] * h->side_h[0] +
                                   (unsigned long long)in_bytes_per_px(h->fmt[1]) * h->side_w[1] * h->side_h[1];
    h->alg_bytes = 120ULL * sum_px + in2 + 72ULL * sum_px_ge1;
    // compulsory I/O floor B_io = in_0 * P_0 + 8
    h->io_bytes = in2 / 2 + 8ULL;
}

// Exact memo of one side's transfer function (Geo::eotf_lut), built by the device code it replaces: the R / B tables of
// 10-bit P016 and NV12 (also those of P216 / YUV444P16 and NV16 / YUV444: the tables are indexed per pixel by (Cr, Y) and
// (Cb, Y), whatever the subsampling), the sRGB16 table.  The other formats (and the deep 16-bit YUV sides) have none.
static cudaError_t build_side_lut(int fmt, bool deep, Geo& g, float** lut, size_t* bytes)
{
    *bytes = 0;
    if (format_is_yuv(fmt) && !deep) {
        const bool b16 = format_is_yuv16(fmt);
        const int n = b16 ? 1024 : 256, shift = b16 ? 6 : 0;
        const size_t b = (size_t)2 * n * n * sizeof(float);
        cudaError_t e = cudaMalloc(lut, b);
        if (e != cudaSuccess) return e;
        k_build_eotf_lut<<<(n * n + 255) / 256, 256>>>(g.coef, n, shift, *lut);
        if ((e = cudaGetLastError()) != cudaSuccess || (e = cudaDeviceSynchronize()) != cudaSuccess) return e;
        g.eotf_lut = *lut;
        g.lut_n = n;
        g.lut_shift = shift;
        *bytes = b;
    }
    if (fmt == kSRGB16) {
        // exact memo of the sRGB16 transfer function: one gather per sample instead of one powf
        const size_t b = (size_t)65536 * sizeof(float);
        cudaError_t e = cudaMalloc(lut, b);
        if (e != cudaSuccess) return e;
        k_build_srgb16_lut<<<65536 / 256, 256>>>(*lut);
        if ((e = cudaGetLastError()) != cudaSuccess || (e = cudaDeviceSynchronize()) != cudaSuccess) return e;
        g.eotf_lut = *lut;
        g.lut_n = 65536;
        g.lut_shift = 0;
        *bytes = b;
    }
    return cudaSuccess;
}

// the distorted description of ssimu2_create_mixed (checked like ssimu2_config, before any device call)
static int check_source(const ssimu2_config* cfg, const ssimu2_source* s)
{
    if (!format_known(s->format)) return SSIMU2_E_UNSUPPORTED;
    if (s->matrix < 0 || s->matrix > 2) return SSIMU2_E_UNSUPPORTED;
    if (s->flags & ~SSIMU2_FLAG_P016_DEEP) return SSIMU2_E_UNSUPPORTED;
    if ((s->flags & SSIMU2_FLAG_P016_DEEP) && !format_is_yuv16(s->format)) return SSIMU2_E_UNSUPPORTED;
    for (int i = 0; i < 2; i++)
        if (s->reserved[i]) return SSIMU2_E_INVALID;
    if ((s->width == 0) != (s->height == 0)) return SSIMU2_E_INVALID;
    // only upscaling: the distorted frames are at most the reference's size on each axis
    if (s->width > cfg->width || s->height > cfg->height) return SSIMU2_E_UNSUPPORTED;
    return SSIMU2_OK;
}

// the distorted frames' size (0, 0: the reference's)
static uint32_t source_width(const ssimu2_config* cfg, const ssimu2_source* s) { return s && s->width ? s->width : cfg->width; }
static uint32_t source_height(const ssimu2_config* cfg, const ssimu2_source* s) { return s && s->height ? s->height : cfg->height; }

// The two sides are one effective description: same format and deep flag, and (YUV) same matrix and range.  Matrix and range
// mean nothing to the packed formats.
static bool same_source(const ssimu2_config* cfg, const ssimu2_source* s)
{
    const bool yuv = format_is_yuv(cfg->format);
    return s->format == cfg->format && (s->flags & SSIMU2_FLAG_P016_DEEP) == (cfg->flags & SSIMU2_FLAG_P016_DEEP) &&
           (!yuv || (s->matrix == cfg->matrix && (s->full_range != 0) == (cfg->full_range != 0))) &&
           source_width(cfg, s) == cfg->width && source_height(cfg, s) == cfg->height;
}

// ---- scaled distorted frames: plane grids, tap tables and the staged layout of k_resample (resample.cuh) ----
// Catmull-Rom (Keys, a = -0.5) weight of a tap at distance t, in double (this file's host code is built with
// -ffp-contract=off: the oracle evaluates the same expressions uncontracted).
static double keys_weight(double t)
{
    if (t < 1.0) return (1.5 * t - 2.5) * t * t + 1.0;
    if (t < 2.0) return ((-0.5 * t + 2.5) * t - 4.0) * t + 2.0;
    return 0.0;
}

// Taps of an axis of `in` -> `out` samples: output coordinate x reads source samples i - 1 .. i + 2 (clamped when read),
// i = floor(sx), sx = (x + 0.5) * in / out - 0.5 (centre-aligned).  An axis of unchanged size gets (0, 1, 0, 0).
static void axis_taps(int in, int out, float4* w, int* j0)
{
    const double scale = (double)in / (double)out;
    for (int x = 0; x < out; x++) {
        const double sx = (x + 0.5) * scale - 0.5;
        const int i = (int)floor(sx);
        float ww[4];
        for (int k = 0; k < 4; k++) ww[k] = (float)keys_weight(fabs(sx - (double)(i - 1 + k)));
        w[x] = make_float4(ww[0], ww[1], ww[2], ww[3]);
        j0[x] = i - 1;
    }
}

// The plane grids of the distorted format at its own size (in) and the reference's (out), the staged layout (NVDEC-like:
// pitch and planes 256-byte aligned; 4:4:4 Cr at plane[1] + (plane[1] - plane[0])) and the tap tables in one device buffer.
static cudaError_t build_resample(ssimu2_handle* h)
{
    const int fmt = h->fmt[1];
    const int W = (int)h->side_w[0], H = (int)h->side_h[0], Wd = (int)h->side_w[1], Hd = (int)h->side_h[1];
    const bool yuv = format_is_yuv(fmt), yuv444 = fmt == kYUV444 || fmt == kYUV444P16, yuv420 = fmt == kNV12 || fmt == kP016;
    const uint64_t s = fmt == kSRGBF32 || fmt == kLINEARF32 ? 4 : (format_is_yuv16(fmt) || fmt == kSRGB16) ? 2 : 1;
    RsArgs& a = h->rs;
    a.nplanes = !yuv ? 1 : yuv444 ? 3 : 2;
    int dims[3][4];   // per plane: in_w, in_h, out_w, out_h (per channel)
    int nch[3] = {yuv ? 1 : 3, yuv444 ? 1 : 2, 1};
    dims[0][0] = Wd; dims[0][1] = Hd; dims[0][2] = W; dims[0][3] = H;
    if (yuv444) {
        for (int p = 1; p < 3; p++) memcpy(dims[p], dims[0], sizeof(dims[0]));
    } else if (yuv) {
        dims[1][0] = (Wd + 1) / 2; dims[1][1] = yuv420 ? (Hd + 1) / 2 : Hd;
        dims[1][2] = (W + 1) / 2;  dims[1][3] = yuv420 ? (H + 1) / 2 : H;
    }
    uint64_t row = (uint64_t)W * nch[0] * s;
    if (yuv) row = std::max<uint64_t>(row, (uint64_t)dims[1][2] * nch[1] * s);
    a.dst_pitch = (uint32_t)((row + 255) / 256 * 256);
    uint64_t off = 0;
    for (int p = 0; p < a.nplanes; p++) {
        a.pl[p].dst_off = (long long)off;
        off += (uint64_t)a.dst_pitch * dims[p][3];
        off = (off + 255) / 256 * 256;
    }
    a.dst_stride = (long long)off;
    // 4:4:4: the front-end finds Cr at plane[1] + (plane[1] - plane[0]), so the three planes must be equally spaced
    if (yuv444 && a.pl[2].dst_off != 2 * a.pl[1].dst_off) return cudaErrorInvalidValue;
    // tap tables: per plane grid, x then y (4:4:4 chroma shares the luma tables)
    std::vector<float4> w;
    std::vector<int> j;
    size_t wofs[3][2], jofs[3][2];
    const int ngrids = yuv444 ? 1 : a.nplanes;
    for (int p = 0; p < ngrids; p++)
        for (int ax = 0; ax < 2; ax++) {
            const int in = dims[p][ax], out = dims[p][2 + ax];
            wofs[p][ax] = w.size();
            jofs[p][ax] = j.size();
            w.resize(w.size() + out);
            j.resize(j.size() + out);
            axis_taps(in, out, &w[wofs[p][ax]], &j[jofs[p][ax]]);
        }
    const size_t wb = w.size() * sizeof(float4), jb = j.size() * sizeof(int);
    cudaError_t e = cudaMalloc(&h->rs_tab, wb + jb);
    if (e != cudaSuccess) return e;
    if ((e = cudaMemcpy(h->rs_tab, w.data(), wb, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
    if ((e = cudaMemcpy((uint8_t*)h->rs_tab + wb, j.data(), jb, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
    h->device_bytes += wb + jb;
    const float4* wd = (const float4*)h->rs_tab;
    const int* jd = (const int*)((uint8_t*)h->rs_tab + wb);
    int tiles = 0;
    for (int p = 0; p < a.nplanes; p++) {
        RsPlane& P = a.pl[p];
        const int g = yuv444 ? 0 : p;
        P.in_w = dims[p][0]; P.in_h = dims[p][1]; P.out_w = dims[p][2]; P.out_h = dims[p][3];
        P.x = RsAxis{wd + wofs[g][0], jd + jofs[g][0]};
        P.y = RsAxis{wd + wofs[g][1], jd + jofs[g][1]};
        P.tiles_x = (P.out_w + kRsTileX - 1) / kRsTileX;
        P.tile0 = tiles;
        tiles += P.tiles_x * ((P.out_h + kRsTileY - 1) / kRsTileY);
    }
    a.tiles = tiles;
    return cudaSuccess;
}

// ---- TMA tensor maps (driver entry point fetched through the runtime; libcuda is not linked) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_plane_map(EncodeTiledFn enc, CUtensorMap* out, float* base, const ScaleDesc& d, int planes, long long slot_stride,
                          uint32_t batch, uint32_t box_cols, uint32_t box_rows, bool swizzle128)
{
    // 4-D view {x, y, plane, frame} of a [frame][plane][h][pitch] f32 buffer; out-of-range elements read as 0
    cuuint64_t dims[4] = {(cuuint64_t)d.w, (cuuint64_t)d.h, (cuuint64_t)planes, (cuuint64_t)batch};
    cuuint64_t strides[3] = {(cuuint64_t)d.pitch * 4, (cuuint64_t)d.h * d.pitch * 4, (cuuint64_t)slot_stride * 4};
    cuuint32_t box[4] = {box_cols, box_rows, (cuuint32_t)planes, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : SSIMU2_E_INTERNAL;
}

static int build_tma_maps(ssimu2_handle* h, Slot& sl)
{
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
        qres != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        return SSIMU2_E_INTERNAL;
    }
    EncodeTiledFn enc = (EncodeTiledFn)fn;
    const Geo& g = h->geo;
    for (int s = 0; s < g.nscales; s++) {
        float* xyb = sl.xyb + g.sc[s].xyb_off;
        int r;
        if (h->pipeline == 0) {
            r = make_plane_map(enc, &sl.maps_x.xyb_in[s], xyb, g.sc[s], 6, g.xyb_stride, h->batch, kXInW, kXR, false);
            if (r) return r;
            continue;
        }
        float* hb = sl.hb + g.sc[s].hb_off;
        r = make_plane_map(enc, &sl.maps.hb[s], hb, g.sc[s], 15, g.hb_stride, h->batch, kVCols, kVRowsPerStage, false);
        if (r) return r;
        r = make_plane_map(enc, &sl.maps.xyb[s], xyb, g.sc[s], 6, g.xyb_stride, h->batch, kVCols, kVRowsPerStage, false);
        if (r) return r;
        r = make_plane_map(enc, &sl.maps_h.xyb_in[s], xyb, g.sc[s], 6, g.xyb_stride, h->batch, kHCols, kHRows, true);
        if (r) return r;
        r = make_plane_map(enc, &sl.maps_h.hb_out[s], hb, g.sc[s], 15, g.hb_stride, h->batch, kHCols, kHRows, true);
        if (r) return r;
    }
    return 0;
}

// ---- launch logic -------------------------------------------------------------------------------
// All work of a batch runs on its slot's stream: [frame-table upload + front-end] x (1 .. n launches), then
// k_hv + k_finalize (or k_hpass + k_vpass + k_finalize), then the D2H copy of scores and norms.

template <int FMT, int SIDE>
static void launch_frontend_kernel(const Geo& g, const FramePair* tab, Slot& sl, uint32_t frame0, uint32_t n)
{
    const int rx = (g.sc[0].w + kF2Region - 1) / kF2Region, ry = (g.sc[0].h + kF2Region - 1) / kF2Region;
    const int per_cta = (kF2Threads / 32) * f2_regions_per_warp(SIDE);
    k_frontend2<FMT, SIDE><<<dim3((rx + per_cta - 1) / per_cta, ry, n), kF2Threads, 0, sl.stream>>>(g, tab, sl.xyb, (int)frame0);
}

// fe_fmt: the front-end format of the side(s) (kP016A / kP216A / kYUV444P16A for a 16-bit YUV side with SSIMU2_FLAG_P016_DEEP);
// tab: the device frame table the launch reads
template <int SIDE>
static int launch_frontend_side(const Geo& g, int fe_fmt, const FramePair* tab, Slot& sl, uint32_t frame0, uint32_t n)
{
    switch (fe_fmt) {
    case kNV12: launch_frontend_kernel<kNV12, SIDE>(g, tab, sl, frame0, n); break;
    case kP016: launch_frontend_kernel<kP016, SIDE>(g, tab, sl, frame0, n); break;
    case kP016A: launch_frontend_kernel<kP016A, SIDE>(g, tab, sl, frame0, n); break;
    case kSRGB8: launch_frontend_kernel<kSRGB8, SIDE>(g, tab, sl, frame0, n); break;
    case kSRGB16: launch_frontend_kernel<kSRGB16, SIDE>(g, tab, sl, frame0, n); break;
    case kSRGBF32: launch_frontend_kernel<kSRGBF32, SIDE>(g, tab, sl, frame0, n); break;
    case kLINEARF32: launch_frontend_kernel<kLINEARF32, SIDE>(g, tab, sl, frame0, n); break;
    case kNV16: launch_frontend_kernel<kNV16, SIDE>(g, tab, sl, frame0, n); break;
    case kP216: launch_frontend_kernel<kP216, SIDE>(g, tab, sl, frame0, n); break;
    case kP216A: launch_frontend_kernel<kP216A, SIDE>(g, tab, sl, frame0, n); break;
    case kYUV444: launch_frontend_kernel<kYUV444, SIDE>(g, tab, sl, frame0, n); break;
    case kYUV444P16: launch_frontend_kernel<kYUV444P16, SIDE>(g, tab, sl, frame0, n); break;
    case kYUV444P16A: launch_frontend_kernel<kYUV444P16A, SIDE>(g, tab, sl, frame0, n); break;
    default: return SSIMU2_E_UNSUPPORTED;
    }
    return 0;
}

template <int FMT>
static void launch_resample_kernel(const RsArgs& a, Slot& sl, uint32_t frame0, uint32_t n)
{
    k_resample<FMT><<<dim3((unsigned)a.tiles, 1, n), kRsThreads, 0, sl.stream>>>(a, sl.in_d, (int)frame0);
}

// upscale the distorted frames of pairs [frame0, frame0 + n) into the slot's rs_frames (staged frame i - frame0 for pair i)
static int launch_resample(const ssimu2_handle* h, Slot& sl, uint32_t frame0, uint32_t n)
{
    RsArgs a = h->rs;
    a.dst = sl.rs_frames;
    switch (h->fmt[1]) {
    case kNV12: launch_resample_kernel<kNV12>(a, sl, frame0, n); break;
    case kP016: launch_resample_kernel<kP016>(a, sl, frame0, n); break;
    case kSRGB8: launch_resample_kernel<kSRGB8>(a, sl, frame0, n); break;
    case kSRGB16: launch_resample_kernel<kSRGB16>(a, sl, frame0, n); break;
    case kSRGBF32: launch_resample_kernel<kSRGBF32>(a, sl, frame0, n); break;
    case kLINEARF32: launch_resample_kernel<kLINEARF32>(a, sl, frame0, n); break;
    case kNV16: launch_resample_kernel<kNV16>(a, sl, frame0, n); break;
    case kP216: launch_resample_kernel<kP216>(a, sl, frame0, n); break;
    case kYUV444: launch_resample_kernel<kYUV444>(a, sl, frame0, n); break;
    case kYUV444P16: launch_resample_kernel<kYUV444P16>(a, sl, frame0, n); break;
    default: return SSIMU2_E_UNSUPPORTED;
    }
    return 0;
}

// front-end of pairs [sl.fe_pairs, upto) of the batch being recorded in `sl`: one launch, or on a mixed handle one per side
// (on a scaled handle with k_resample between the two)
static int launch_frontend(ssimu2_handle* h, Slot& sl, uint32_t upto, bool time_it)
{
    const uint32_t f0 = sl.fe_pairs;
    if (upto <= f0) return 0;
    const uint32_t n = upto - f0;
    if (sl.have_dep) {
        // ordered after everything the submitter had enqueued on its stream when it submitted these pairs
        CU_TRY(cudaStreamWaitEvent(sl.stream, sl.ev_in, 0));
        sl.have_dep = false;
    }
    CU_TRY(cudaMemcpyAsync(sl.in_d + f0, sl.in_h + f0, (size_t)n * sizeof(FramePair), cudaMemcpyHostToDevice, sl.stream));
    if (h->scaled) {
        // the distorted front-end reads the upscaled frames: staged frame i - f0 for pair i (plane layout of h->rs)
        if (n > h->rs_group) return SSIMU2_E_INTERNAL;
        for (uint32_t i = f0; i < upto; i++) {
            uint8_t* d = sl.rs_frames + (size_t)(i - f0) * h->rs.dst_stride;
            sl.rs_in_h[i] = sl.in_h[i];
            sl.rs_in_h[i].dis.p0 = d;
            sl.rs_in_h[i].dis.p1 = h->rs.nplanes > 1 ? d + h->rs.pl[1].dst_off : nullptr;
            sl.rs_in_h[i].dis.pitch = h->rs.dst_pitch;
            sl.rs_in_h[i].dis.pad = 0;
        }
        CU_TRY(cudaMemcpyAsync(sl.rs_in_d + f0, sl.rs_in_h + f0, (size_t)n * sizeof(FramePair), cudaMemcpyHostToDevice, sl.stream));
    }
    if (time_it) cudaEventRecord(sl.ev_k[0], sl.stream);
    int r;
    if (!h->mixed) {
        r = launch_frontend_side<kF2Both>(h->geo, h->fe_fmt[0], sl.in_d, sl, f0, n);
    } else {
        r = launch_frontend_side<kF2Ref>(h->geo, h->fe_fmt[0], sl.in_d, sl, f0, n);
        if (!r && h->scaled) r = launch_resample(h, sl, f0, n);
        if (!r) r = launch_frontend_side<kF2Dis>(h->geo_dis, h->fe_fmt[1], h->scaled ? sl.rs_in_d : sl.in_d, sl, f0, n);
    }
    if (r) return r;
    // the timing mark and the "inputs consumed" event follow the last launch: both sides have been read
    if (time_it) cudaEventRecord(sl.ev_k[1], sl.stream);
    CU_TRY(cudaGetLastError());
    h->launches += !h->mixed ? 1 : h->scaled ? 3 : 2;
    if (sl.fe_launches >= sl.ev_fe.size()) {
        cudaEvent_t e = nullptr;
        CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        sl.ev_fe.push_back(e);
    }
    CU_TRY(cudaEventRecord(sl.ev_fe[sl.fe_launches], sl.stream));
    for (uint32_t i = f0; i < upto; i++) sl.fe_seq[i] = (uint16_t)sl.fe_launches;
    sl.fe_launches++;
    sl.fe_pairs = upto;
    return 0;
}

// launch the batch recorded in slot si (it must hold at least one pair and not be launched yet)
static int launch_batch(ssimu2_handle* h, int si)
{
    Slot& sl = h->slots[si];
    if (sl.count == 0 || sl.inflight) return 0;
    const Geo& g = h->geo;
    const uint32_t n = sl.count;
    cudaStream_t st = sl.stream;
    // per-kernel timing is only meaningful when the whole batch goes through one front-end launch
    const bool timed = sl.timed && sl.fe_pairs == 0;
    int r = launch_frontend(h, sl, n, timed);
    if (r) return r;
    if (h->pipeline == 0) {
        HvArgs a{};
        a.hstate = sl.hstate;
        a.flags = sl.hvflags;
        a.ticket = sl.hvflags + (size_t)h->batch * g.total_recs;
        a.partials = sl.partials;
        a.epoch = ++sl.epoch;
        a.nframes = (int)n;
        a.lite_bits = 0;
        for (int s = 0; s < kMaxScales; s++) a.lite_bits |= (uint32_t)(h->lite[s] & 7u) << (4 * s);
        a.tiles = sl.tiles;
        a.tile_log2 = h->tile_log2;
        if (timed) cudaEventRecord(sl.ev_k[2], st);
        if (h->tile)
            k_hv<true><<<(unsigned)(g.items_v * n), kXThreads, kXSmemBytes, st>>>(g, sl.maps_x, a);
        else
            k_hv<false><<<(unsigned)(g.items_v * n), kXThreads, kXSmemBytes, st>>>(g, sl.maps_x, a);
        if (timed) cudaEventRecord(sl.ev_k[3], st);
        k_finalize<<<n, 128, 0, st>>>(g, sl.partials, sl.norms_d, h->scores_ring_d, sl.first_ticket, kResultCap, sl.scores_d, a.ticket);
        if (h->tile) k_tile_finalize<<<dim3(h->tiles_x * h->tiles_y, n), 128, 0, st>>>(g, sl.tiles, h->tile_log2, sl.tile_scores_d);
        if (timed) cudaEventRecord(sl.ev_k[4], st);
        h->launches += h->tile ? 3 : 2;
    } else {
        k_hpass<<<dim3(g.items_h, n), kHThreads, kHSmemBytes, st>>>(g, sl.maps_h);
        if (timed) cudaEventRecord(sl.ev_k[2], st);
        k_vpass<<<dim3(g.items_v, n), kVTmaThreads, kVSmemBytes, st>>>(g, sl.maps, sl.partials);
        if (timed) cudaEventRecord(sl.ev_k[3], st);
        k_finalize<<<n, 128, 0, st>>>(g, sl.partials, sl.norms_d, h->scores_ring_d, sl.first_ticket, kResultCap, sl.scores_d, nullptr);
        if (timed) cudaEventRecord(sl.ev_k[4], st);
        h->launches += 3;
    }
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(sl.scores_h, sl.scores_d, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (!h->score_only)
        CU_TRY(cudaMemcpyAsync(sl.norms_h, sl.norms_d, (size_t)n * 108 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (h->tile)
        CU_TRY(cudaMemcpyAsync(sl.tile_scores_h, sl.tile_scores_d, (size_t)n * h->tiles_x * h->tiles_y * sizeof(double),
                               cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaEventRecord(sl.ev_done, st));
    sl.inflight = true;
    sl.was_timed = timed;
    return 0;
}

// wait for a launched slot and move its results into the ticket-indexed host rings
static int harvest(ssimu2_handle* h, uint32_t si)
{
    Slot& sl = h->slots[si];
    if (!sl.inflight) return 0;
    CU_TRY(cudaEventSynchronize(sl.ev_done));
    for (uint32_t i = 0; i < sl.count; i++) {
        uint64_t t = sl.first_ticket + i, r = t % kResultCap;
        h->res_scores[r] = sl.scores_h[i];
        if (!h->score_only) memcpy(&h->res_norms[r * 108], &sl.norms_h[(size_t)i * 108], 108 * sizeof(double));
        h->res_slot[r] = (int32_t)si;
        if (h->tile) {
            const size_t nt = (size_t)h->tiles_x * h->tiles_y;
            memcpy(&h->res_tiles[(t % h->tile_cap) * nt], &sl.tile_scores_h[i * nt], nt * sizeof(double));
        }
    }
    if (sl.was_timed) {
        // fused: front-end [0,1], k_hv [2,3], (no separate V pass), finalize [3,4]; split: front-end [0,1], H [1,2], V [2,3], finalize [3,4]
        static const int fa[4] = {0, 2, 3, 3}, fb[4] = {1, 3, 3, 4}, sa[4] = {0, 1, 2, 3}, sb[4] = {1, 2, 3, 4};
        for (int k = 0; k < 4; k++) {
            const int a = h->pipeline == 0 ? fa[k] : sa[k], b = h->pipeline == 0 ? fb[k] : sb[k];
            h->last_ms[k] = 0.f;
            if (a != b) cudaEventElapsedTime(&h->last_ms[k], sl.ev_k[a], sl.ev_k[b]);
            h->total_ms[k] += h->last_ms[k];
        }
        h->timed_batches++;
        h->timed_pairs += sl.count;
    }
    sl.inflight = false;
    sl.count = 0;
    sl.fe_pairs = 0;
    sl.fe_launches = 0;
    return 0;
}

// make slot `cur` ready to record a pair
static int prepare_cur(ssimu2_handle* h)
{
    Slot& sl = h->slots[h->cur];
    if (sl.inflight) {
        int r = harvest(h, h->cur);
        if (r) return r;
    }
    if (sl.count == 0) {
        sl.first_ticket = h->next_ticket;
        sl.have_dep = false;
        sl.dep_stream = nullptr;
    }
    return 0;
}

static int finish_pair(ssimu2_handle* h)
{
    Slot& sl = h->slots[h->cur];
    sl.count++;
    h->next_ticket++;
    if (sl.count == h->batch) {
        int r = launch_batch(h, (int)h->cur);
        if (r) return r;
        h->cur = (h->cur + 1) % h->ring;
    } else if (h->input_group && sl.count - sl.fe_pairs >= h->input_group) {
        return launch_frontend(h, sl, sl.count, false);
    }
    return 0;
}

static bool is_yuv(int fmt) { return format_is_yuv(fmt); }

// side 0: a reference frame, 1: a distorted frame (each side is checked against its own format); host frames with the byte
// count copied from plane[0]
static bool frame_ok(const ssimu2_handle* h, const ssimu2_frame* f, int side, bool host = false, size_t bytes = 0)
{
    return frame_layout_ok(h->fmt[side], h->side_w[side], h->side_h[side], f, host, bytes);
}

// locate a ticket: 0 = results on host, 1 = in a launched slot, 2 = in the slot being filled
static int locate(ssimu2_handle* h, uint64_t ticket, uint32_t* slot_out)
{
    if (ticket >= h->next_ticket) return -1;
    if (h->next_ticket - ticket > kResultCap) return -1;
    for (uint32_t i = 0; i < h->ring; i++) {
        Slot& sl = h->slots[i];
        if (sl.count && ticket >= sl.first_ticket && ticket < sl.first_ticket + sl.count) {
            *slot_out = i;
            return sl.inflight ? 1 : 2;
        }
    }
    return 0;
}

// the slot that holds `ticket`, launched if it was still being filled; where = 0 when the results are already on the host
static int locate_launched(ssimu2_handle* h, uint64_t ticket, uint32_t* si, int* where)
{
    *where = locate(h, ticket, si);
    if (*where < 0) return SSIMU2_E_TICKET;
    if (*where == 2) {
        int r = launch_batch(h, (int)*si);
        if (r) return r;
        if (*si == h->cur) h->cur = (h->cur + 1) % h->ring;
        *where = 1;
    }
    return 0;
}

// record the submitter's stream as a dependency of the input group being recorded
static int note_dependency(Slot& sl, void* stream)
{
    if ((cudaStream_t)stream == sl.stream) return 0;
    if (sl.have_dep && sl.dep_stream != stream) {
        // the submitter switched streams inside one input group: pin the dependency on the previous stream now
        CU_TRY(cudaStreamWaitEvent(sl.stream, sl.ev_in, 0));
    }
    CU_TRY(cudaEventRecord(sl.ev_in, (cudaStream_t)stream));
    sl.dep_stream = stream;
    sl.have_dep = true;
    return 0;
}

// one host pair: copy each frame (its own byte count) to the slot's staging ring and record the pair
static int submit_host_pair(ssimu2_handle* h, const ssimu2_frame* ref, size_t ref_bytes, const ssimu2_frame* dis, size_t dis_bytes)
{
    if (!frame_ok(h, ref, 0, true, ref_bytes) || !frame_ok(h, dis, 1, true, dis_bytes)) return SSIMU2_E_INVALID;
    const bool yuv_ref = is_yuv(h->fmt[0]), yuv_dis = is_yuv(h->fmt[1]);
    DeviceGuard guard(h->cfg.device);
    const size_t frame_bytes = ref_bytes > dis_bytes ? ref_bytes : dis_bytes;
    if (frame_bytes > h->staging_frame_bytes) {
        // (re)allocate the staging rings; rare (first call), so a full drain is acceptable
        int fr = ssimu2_flush(h);
        if (fr) return fr;
        for (uint32_t i = 0; i < h->ring; i++) {
            int r = harvest(h, i);
            if (r) return r;
        }
        size_t fb = (frame_bytes + 255) / 256 * 256;
        for (auto& sl : h->slots) {
            cudaFree(sl.staging);
            sl.staging = nullptr;
            if (cudaMalloc(&sl.staging, fb * 2 * h->batch) != cudaSuccess) { cudaGetLastError(); return SSIMU2_E_NOMEM; }
        }
        h->device_bytes += (fb - h->staging_frame_bytes) * 2 * h->batch * h->ring;
        h->staging_frame_bytes = fb;
    }
    int r = prepare_cur(h);
    if (r) return r;
    Slot& sl = h->slots[h->cur];
    uint8_t* da = sl.staging + (size_t)(2 * sl.count) * h->staging_frame_bytes;
    uint8_t* db = da + h->staging_frame_bytes;
    CU_TRY(cudaMemcpyAsync(da, (const void*)ref->plane[0], ref_bytes, cudaMemcpyHostToDevice, sl.stream));
    CU_TRY(cudaMemcpyAsync(db, (const void*)dis->plane[0], dis_bytes, cudaMemcpyHostToDevice, sl.stream));
    FramePair& fp = sl.in_h[sl.count];
    fp.ref.p0 = da; fp.ref.p1 = yuv_ref ? da + (ref->plane[1] - ref->plane[0]) : nullptr; fp.ref.pitch = ref->pitch; fp.ref.pad = 0;
    fp.dis.p0 = db; fp.dis.p1 = yuv_dis ? db + (dis->plane[1] - dis->plane[0]) : nullptr; fp.dis.pitch = dis->pitch; fp.dis.pad = 0;
    return finish_pair(h);
}

}  // namespace

extern "C" {

uint32_t ssimu2_version(void) { return (2u << 16) | 3u; }

const char* ssimu2_strerror(int status)
{
    switch (status) {
    case SSIMU2_OK: return "ok";
    case SSIMU2_E_INVALID: return "invalid argument";
    case SSIMU2_E_UNSUPPORTED: return "unsupported format, size or mode";
    case SSIMU2_E_NOMEM: return "out of memory";
    case SSIMU2_E_NODEVICE: return "no usable CUDA device (sm_100 required)";
    case SSIMU2_E_TICKET: return "unknown or expired ticket";
    case SSIMU2_E_INTERNAL: return "internal error";
    }
    if (status > 0) return cudaGetErrorString((cudaError_t)status);
    return "unknown status";
}

int ssimu2_create(ssimu2_t** out, const ssimu2_config* cfg) { return ssimu2_create_mixed(out, cfg, nullptr); }

int ssimu2_create_mixed(ssimu2_t** out, const ssimu2_config* cfg, const ssimu2_source* dis)
{
    if (!out || !cfg) return SSIMU2_E_INVALID;
    *out = nullptr;
    if (cfg->width < 8 || cfg->height < 8 || cfg->width > 32768 || cfg->height > 32768) return SSIMU2_E_UNSUPPORTED;
    if (!format_known(cfg->format)) return SSIMU2_E_UNSUPPORTED;
    if (cfg->matrix < 0 || cfg->matrix > 2) return SSIMU2_E_UNSUPPORTED;
    if (cfg->pipeline > SSIMU2_PIPELINE_SPLIT) return SSIMU2_E_UNSUPPORTED;
    if (cfg->flags & ~(SSIMU2_FLAG_SCORE_ONLY | SSIMU2_FLAG_NO_TIMING | SSIMU2_FLAG_P016_DEEP)) return SSIMU2_E_UNSUPPORTED;
    if ((cfg->flags & SSIMU2_FLAG_P016_DEEP) && !format_is_yuv16(cfg->format)) return SSIMU2_E_UNSUPPORTED;
    if ((cfg->flags & SSIMU2_FLAG_SCORE_ONLY) && cfg->pipeline != SSIMU2_PIPELINE_DEFAULT) return SSIMU2_E_UNSUPPORTED;
    for (int i = 0; i < 4; i++)
        if (cfg->reserved[i]) return SSIMU2_E_INVALID;
    if (cfg->tile && (cfg->tile < 64 || cfg->tile > 32768 || (cfg->tile & (cfg->tile - 1)) ||
                      cfg->pipeline != SSIMU2_PIPELINE_DEFAULT))
        return SSIMU2_E_UNSUPPORTED;
    if (dis) {
        const int rc = check_source(cfg, dis);
        if (rc) return rc;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        return SSIMU2_E_NODEVICE;
    }
    if (cfg->device < 0 || cfg->device >= ndev) return SSIMU2_E_INVALID;
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    // the only SASS in this library is sm_100a; architecture-specific targets are not forward compatible (sm_103 cannot run it)
    if (prop.major != 10 || prop.minor != 0) return SSIMU2_E_NODEVICE;

    ssimu2_handle* h = new (std::nothrow) ssimu2_handle();
    if (!h) return SSIMU2_E_NOMEM;
    h->cfg = *cfg;
    h->mixed = dis != nullptr && !same_source(cfg, dis);
    h->side_w[0] = cfg->width;
    h->side_h[0] = cfg->height;
    h->side_w[1] = source_width(cfg, dis);
    h->side_h[1] = source_height(cfg, dis);
    h->scaled = h->side_w[1] != cfg->width || h->side_h[1] != cfg->height;
    const bool deep_ref = (cfg->flags & SSIMU2_FLAG_P016_DEEP) != 0;
    // upscaled 16-bit samples generally have non-zero low bits: a scaled 16-bit YUV side always takes the deep front-end (the
    // same bits as the memo path, which would send most samples to its arithmetic fall-back anyway)
    const bool deep_dis = h->mixed ? (dis->flags & SSIMU2_FLAG_P016_DEEP) != 0 || (h->scaled && format_is_yuv16(dis->format))
                                   : deep_ref;
    h->fmt[0] = cfg->format;
    h->fmt[1] = h->mixed ? dis->format : cfg->format;
    h->fe_fmt[0] = deep_ref ? deep_fe_fmt(h->fmt[0]) : h->fmt[0];
    h->fe_fmt[1] = deep_dis ? deep_fe_fmt(h->fmt[1]) : h->fmt[1];
    h->ring = cfg->ring ? cfg->ring : kDefaultRing;
    if (h->ring > 16) h->ring = 16;
    h->batch = cfg->batch ? cfg->batch : kDefaultBatch;
    if (h->batch > (uint32_t)kMaxBatch) h->batch = kMaxBatch;
    h->input_group = cfg->input_group >= h->batch ? 0 : cfg->input_group;
    h->pipeline = (int)cfg->pipeline;
    h->score_only = (cfg->flags & SSIMU2_FLAG_SCORE_ONLY) != 0;
    build_geo(h);
    if (cfg->batch == 0) {
        // default batch: enough k_hv work items (64-column strips over all scales) for ~8 waves of one CTA per SM, as a power
        // of two, while the workspace of all ring slots stays under 8 GiB (4K: 8 pairs, 1080p: 32, 512x512: 128)
        const uint64_t per_pair = (uint64_t)h->geo.xyb_stride * 4 + (uint64_t)h->geo.total_recs * kXHsBytes;
        uint32_t b = kDefaultBatch;
        while (b < 256 && (uint64_t)b * h->geo.items_v < 8u * 148u) b *= 2;
        while (b > kDefaultBatch && (uint64_t)b * h->ring * per_pair > (8ull << 30)) b /= 2;
        h->batch = b;
    }
    if (h->score_only) {
        // a channel of a scale is "lite" when both of its SSIM' weights are zero; the weight cursor is dense over the scales
        // that exist (k_finalize, cpu.rs:842-854): weight index ((c * nscales + s) * 2 + n) * 3 + map
        static const double w108[108] = {SSIMU2_WEIGHTS108};
        const int ns = h->geo.nscales;
        for (int s = 0; s < ns; s++)
            for (int c = 0; c < 3; c++) {
                const int base = (c * ns + s) * 6;
                if (w108[base + 0] == 0.0 && w108[base + 3] == 0.0) h->lite[s] |= (unsigned char)(1u << c);
            }
    }
    if (cfg->tile) {
        h->tile = cfg->tile;
        while ((1u << h->tile_log2) < cfg->tile) h->tile_log2++;
        h->tiles_x = (cfg->width + cfg->tile - 1) / cfg->tile;
        h->tiles_y = (cfg->height + cfg->tile - 1) / cfg->tile;
        int none;
        h->tile_entries = (size_t)tile_layout(h->geo, h->tile_log2, h->geo.nscales, &none);
        // the host keeps the maps of the last tile_cap tickets (at least four rings' worth of batches), at most ~256 MiB of them
        const uint64_t map_bytes = (uint64_t)h->tiles_x * h->tiles_y * sizeof(double);
        const uint64_t want = std::max<uint64_t>(1024, 4ull * h->batch * h->ring);
        h->tile_cap = std::max<uint64_t>((uint64_t)h->batch * h->ring, std::min<uint64_t>(want, (256ull << 20) / map_bytes));
    }
    DeviceGuard guard(cfg->device);
    int rc = 0;
#define CR(expr)                                  \
    do {                                          \
        cudaError_t _e = (expr);                  \
        if (_e != cudaSuccess) {                  \
            cudaGetLastError();                   \
            rc = (_e == cudaErrorMemoryAllocation) ? SSIMU2_E_NOMEM : (int)_e; \
            goto fail;                            \
        }                                         \
    } while (0)
    try {
        h->slots.resize(h->ring);
        h->res_scores.assign(kResultCap, 0.0);
        h->res_norms.assign(kResultCap * 108, 0.0);
        h->res_slot.assign(kResultCap, -1);
        h->res_tiles.assign((size_t)h->tile_cap * h->tiles_x * h->tiles_y, 0.0);
        for (auto& sl : h->slots) sl.fe_seq.assign(h->batch, 0);
    } catch (...) {
        rc = SSIMU2_E_NOMEM;
        goto fail;
    }
    CR(cudaMalloc(&h->scores_ring_d, kResultCap * sizeof(double)));
    CR(cudaMemset(h->scores_ring_d, 0, kResultCap * sizeof(double)));
    h->device_bytes += kResultCap * sizeof(double);
    CR(cudaFuncSetAttribute((const void*)k_hpass, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHSmemBytes));
    CR(cudaFuncSetAttribute((const void*)k_vpass, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVSmemBytes));
    CR(cudaFuncSetAttribute((const void*)k_hv<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXSmemBytes));
    if (h->tile) CR(cudaFuncSetAttribute((const void*)k_hv<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXSmemBytes));
    {
        exact_math::CbrtScale cs;
        for (int i = 0; i < 256; i++) cs.tab[i] = exact_math::cbrt_scale_entry(i);
        CR(cudaMemcpyToSymbol(kCbrtC, &cs, sizeof(cs)));
    }
    {
        size_t bytes = 0;
        CR(build_side_lut(h->fmt[0], deep_ref, h->geo, &h->eotf_lut, &bytes));
        h->device_bytes += bytes;
    }
    if (h->mixed) {
        // the distorted side: same geometry, its own coefficients and memo table
        size_t bytes = 0;
        h->geo_dis = h->geo;
        h->geo_dis.coef = make_coef(dis->format, dis->matrix, dis->full_range);
        h->geo_dis.eotf_lut = nullptr;
        h->geo_dis.lut_n = h->geo_dis.lut_shift = 0;
        CR(build_side_lut(h->fmt[1], deep_dis, h->geo_dis, &h->eotf_lut_dis, &bytes));
        h->device_bytes += bytes;
    }
    if (h->scaled) {
        CR(build_resample(h));
        h->rs_group = h->input_group ? h->input_group : h->batch;
    }
    for (uint32_t i = 0; i < h->ring; i++) {
        Slot& sl = h->slots[i];
        const Geo& g = h->geo;
        size_t xyb_b = (size_t)g.xyb_stride * h->batch * sizeof(float);
        size_t hb_b = h->pipeline == 0 ? 0 : (size_t)g.hb_stride * h->batch * sizeof(float);
        size_t hs_b = h->pipeline == 0 ? (size_t)g.total_recs * h->batch * kXHsBytes : 0;
        size_t fl_b = h->pipeline == 0 ? ((size_t)g.total_recs * h->batch + 2) * sizeof(uint32_t) : 0;
        size_t part_b = (size_t)g.total_strips * 18 * h->batch * sizeof(double);
        size_t in_b = (size_t)h->batch * sizeof(FramePair);
        CR(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
        CR(cudaEventCreateWithFlags(&sl.ev_in, cudaEventDisableTiming));
        CR(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
        for (int k = 0; k < 5; k++) CR(cudaEventCreate(&sl.ev_k[k]));
        CR(cudaMalloc(&sl.xyb, xyb_b));
        if (hb_b) CR(cudaMalloc(&sl.hb, hb_b));
        if (hs_b) {
            CR(cudaMalloc(&sl.hstate, hs_b));
            CR(cudaMalloc(&sl.hvflags, fl_b));
            CR(cudaMemset(sl.hvflags, 0, fl_b));
        }
        CR(cudaMalloc(&sl.partials, part_b));
        CR(cudaMemset(sl.partials, 0, part_b));
        CR(cudaMalloc(&sl.norms_d, (size_t)h->batch * 108 * sizeof(double)));
        CR(cudaMalloc(&sl.scores_d, (size_t)h->batch * sizeof(double)));
        CR(cudaMalloc(&sl.in_d, in_b));
        CR(cudaMallocHost(&sl.in_h, in_b));
        CR(cudaMallocHost(&sl.norms_h, (size_t)h->batch * 108 * sizeof(double)));
        CR(cudaMallocHost(&sl.scores_h, (size_t)h->batch * sizeof(double)));
        h->device_bytes += xyb_b + hb_b + hs_b + fl_b + part_b + in_b + (size_t)h->batch * 109 * sizeof(double);
        if (h->tile) {
            // every entry k_hv<true> owns is rewritten per batch; the SSIM' entries of X and B of a score-only handle's lite
            // strips are never written and stay 0
            const size_t tab_b = h->tile_entries * 18 * h->batch * sizeof(double);
            const size_t ts_b = (size_t)h->tiles_x * h->tiles_y * h->batch * sizeof(double);
            CR(cudaMalloc(&sl.tiles, tab_b));
            CR(cudaMemset(sl.tiles, 0, tab_b));
            CR(cudaMalloc(&sl.tile_scores_d, ts_b));
            CR(cudaMallocHost(&sl.tile_scores_h, ts_b));
            h->device_bytes += tab_b + ts_b;
        }
        if (h->scaled) {
            const size_t rs_b = (size_t)h->rs_group * h->rs.dst_stride;
            CR(cudaMalloc(&sl.rs_frames, rs_b));
            CR(cudaMalloc(&sl.rs_in_d, in_b));
            CR(cudaMallocHost(&sl.rs_in_h, in_b));
            h->device_bytes += rs_b + in_b;
        }
        rc = build_tma_maps(h, sl);
        if (rc) goto fail;
        sl.timed = (cfg->flags & SSIMU2_FLAG_NO_TIMING) == 0;
    }
    CR(cudaDeviceSynchronize());
    *out = h;
    return SSIMU2_OK;
fail:
    ssimu2_destroy(h);
    return rc;
#undef CR
}

int ssimu2_destroy(ssimu2_t* h)
{
    if (!h) return SSIMU2_OK;
    DeviceGuard guard(h->cfg.device);
    for (auto& sl : h->slots) {
        if (sl.stream) cudaStreamSynchronize(sl.stream);
        if (sl.ev_in) cudaEventDestroy(sl.ev_in);
        if (sl.ev_done) cudaEventDestroy(sl.ev_done);
        for (int k = 0; k < 5; k++)
            if (sl.ev_k[k]) cudaEventDestroy(sl.ev_k[k]);
        for (cudaEvent_t e : sl.ev_fe) cudaEventDestroy(e);
        cudaFree(sl.xyb); cudaFree(sl.hb); cudaFree(sl.hstate); cudaFree(sl.hvflags); cudaFree(sl.partials);
        cudaFree(sl.norms_d); cudaFree(sl.scores_d); cudaFree(sl.staging); cudaFree(sl.in_d);
        cudaFree(sl.rs_frames); cudaFree(sl.rs_in_d); cudaFree(sl.tiles); cudaFree(sl.tile_scores_d);
        if (sl.tile_scores_h) cudaFreeHost(sl.tile_scores_h);
        if (sl.in_h) cudaFreeHost(sl.in_h);
        if (sl.rs_in_h) cudaFreeHost(sl.rs_in_h);
        if (sl.norms_h) cudaFreeHost(sl.norms_h);
        if (sl.scores_h) cudaFreeHost(sl.scores_h);
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    cudaFree(h->scores_ring_d);
    cudaFree(h->eotf_lut);
    cudaFree(h->eotf_lut_dis);
    cudaFree(h->rs_tab);
    delete h;
    return SSIMU2_OK;
}

int ssimu2_mem_usage(const ssimu2_t* h, size_t* bytes)
{
    if (!h || !bytes) return SSIMU2_E_INVALID;
    *bytes = h->device_bytes;
    return SSIMU2_OK;
}

int ssimu2_submit(ssimu2_t* h, const ssimu2_frame* ref, const ssimu2_frame* dis, void* stream, uint64_t* ticket)
{
    if (!h || !frame_ok(h, ref, 0) || !frame_ok(h, dis, 1)) return SSIMU2_E_INVALID;
    DeviceGuard guard(h->cfg.device);
    int r = prepare_cur(h);
    if (r) return r;
    Slot& sl = h->slots[h->cur];
    r = note_dependency(sl, stream);
    if (r) return r;
    FramePair& fp = sl.in_h[sl.count];
    fp.ref.p0 = (const uint8_t*)ref->plane[0]; fp.ref.p1 = (const uint8_t*)ref->plane[1]; fp.ref.pitch = ref->pitch; fp.ref.pad = 0;
    fp.dis.p0 = (const uint8_t*)dis->plane[0]; fp.dis.p1 = (const uint8_t*)dis->plane[1]; fp.dis.pitch = dis->pitch; fp.dis.pad = 0;
    if (ticket) *ticket = h->next_ticket;
    return finish_pair(h);
}

int ssimu2_submit_batch(ssimu2_t* h, uint32_t n, const ssimu2_frame* refs, const ssimu2_frame* diss, void* stream,
                        uint64_t* first_ticket)
{
    if (!h || (n && (!refs || !diss))) return SSIMU2_E_INVALID;
    // all or nothing: every pair is checked before the first one is queued
    for (uint32_t i = 0; i < n; i++)
        if (!frame_ok(h, &refs[i], 0) || !frame_ok(h, &diss[i], 1)) return SSIMU2_E_INVALID;
    if (first_ticket) *first_ticket = h->next_ticket;
    for (uint32_t i = 0; i < n; i++) {
        int r = ssimu2_submit(h, &refs[i], &diss[i], stream, nullptr);
        if (r) return r;
    }
    return SSIMU2_OK;
}

int ssimu2_submit_host(ssimu2_t* h, const ssimu2_frame* ref, const ssimu2_frame* dis, size_t frame_bytes, uint64_t* ticket)
{
    return ssimu2_submit_host_batch(h, 1, ref, dis, frame_bytes, ticket);
}

int ssimu2_submit_host_batch(ssimu2_t* h, uint32_t n, const ssimu2_frame* refs, const ssimu2_frame* diss, size_t frame_bytes,
                             uint64_t* first_ticket)
{
    // one byte count for both frames: only meaningful when the two sides have the same bytes per pixel
    if (h && in_bytes_per_px(h->fmt[0]) != in_bytes_per_px(h->fmt[1])) return SSIMU2_E_INVALID;
    return ssimu2_submit_host_sized(h, n, refs, frame_bytes, diss, frame_bytes, first_ticket);
}

int ssimu2_submit_host_sized(ssimu2_t* h, uint32_t n, const ssimu2_frame* refs, size_t ref_bytes, const ssimu2_frame* diss,
                             size_t dis_bytes, uint64_t* first_ticket)
{
    if (!h || (n && (!refs || !diss))) return SSIMU2_E_INVALID;
    for (uint32_t i = 0; i < n; i++)
        if (!frame_ok(h, &refs[i], 0, true, ref_bytes) || !frame_ok(h, &diss[i], 1, true, dis_bytes)) return SSIMU2_E_INVALID;
    if (first_ticket) *first_ticket = h->next_ticket;
    for (uint32_t i = 0; i < n; i++) {
        int r = submit_host_pair(h, &refs[i], ref_bytes, &diss[i], dis_bytes);
        if (r) return r;
    }
    return SSIMU2_OK;
}

int ssimu2_flush(ssimu2_t* h)
{
    if (!h) return SSIMU2_E_INVALID;
    DeviceGuard guard(h->cfg.device);
    Slot& sl = h->slots[h->cur];
    if (sl.count && !sl.inflight) {
        int r = launch_batch(h, (int)h->cur);
        if (r) return r;
        h->cur = (h->cur + 1) % h->ring;
    }
    return SSIMU2_OK;
}

int ssimu2_wait(ssimu2_t* h, uint64_t ticket)
{
    if (!h) return SSIMU2_E_INVALID;
    DeviceGuard guard(h->cfg.device);
    uint32_t si = 0;
    int where = 0;
    int r = locate_launched(h, ticket, &si, &where);
    if (r) return r;
    if (where == 1) return harvest(h, si);
    return SSIMU2_OK;
}

int ssimu2_completed(ssimu2_t* h, uint64_t* watermark)
{
    if (!h || !watermark) return SSIMU2_E_INVALID;
    uint64_t w = h->next_ticket;
    for (const Slot& sl : h->slots)
        if (sl.count && sl.first_ticket < w) w = sl.first_ticket;
    *watermark = w;
    return SSIMU2_OK;
}

int ssimu2_get_score(ssimu2_t* h, uint64_t ticket, double* score)
{
    if (!h || !score) return SSIMU2_E_INVALID;
    int r = ssimu2_wait(h, ticket);
    if (r) return r;
    *score = h->res_scores[ticket % kResultCap];
    return SSIMU2_OK;
}

int ssimu2_get_scores(ssimu2_t* h, uint64_t first_ticket, uint32_t n, double* scores)
{
    if (!h || (n && !scores)) return SSIMU2_E_INVALID;
    for (uint32_t i = 0; i < n; i++) {
        int r = ssimu2_wait(h, first_ticket + i);
        if (r) return r;
        scores[i] = h->res_scores[(first_ticket + i) % kResultCap];
    }
    return SSIMU2_OK;
}

int ssimu2_get_norms(ssimu2_t* h, uint64_t ticket, double* norms108)
{
    if (!h || !norms108) return SSIMU2_E_INVALID;
    if (h->score_only) return SSIMU2_E_UNSUPPORTED;
    int r = ssimu2_wait(h, ticket);
    if (r) return r;
    memcpy(norms108, &h->res_norms[(ticket % kResultCap) * 108], 108 * sizeof(double));
    return SSIMU2_OK;
}

int ssimu2_compute_sync(ssimu2_t* h, const ssimu2_frame* ref, const ssimu2_frame* dis, void* stream, double* score)
{
    uint64_t t = 0;
    int r = ssimu2_submit(h, ref, dis, stream, &t);
    if (r) return r;
    return ssimu2_get_score(h, t, score);
}

int ssimu2_stream_wait(ssimu2_t* h, uint64_t ticket, void* stream)
{
    if (!h) return SSIMU2_E_INVALID;
    DeviceGuard guard(h->cfg.device);
    uint32_t si = 0;
    int where = 0;
    int r = locate_launched(h, ticket, &si, &where);
    if (r) return r;
    if (where == 1) CU_TRY(cudaStreamWaitEvent((cudaStream_t)stream, h->slots[si].ev_done, 0));
    return SSIMU2_OK;
}

int ssimu2_stream_wait_input(ssimu2_t* h, uint64_t ticket, void* stream)
{
    if (!h) return SSIMU2_E_INVALID;
    DeviceGuard guard(h->cfg.device);
    uint32_t si = 0;
    const int where = locate(h, ticket, &si);
    if (where < 0) return SSIMU2_E_TICKET;
    if (where == 0) return SSIMU2_OK;   // completed long ago
    Slot& sl = h->slots[si];
    const uint32_t idx = (uint32_t)(ticket - sl.first_ticket);
    if (idx >= sl.fe_pairs) {
        // still waiting in an input group: launch the front-end for everything recorded so far
        int r = launch_frontend(h, sl, sl.count, false);
        if (r) return r;
    }
    CU_TRY(cudaStreamWaitEvent((cudaStream_t)stream, sl.ev_fe[sl.fe_seq[idx]], 0));
    return SSIMU2_OK;
}

int ssimu2_get_tile_grid(const ssimu2_t* h, uint32_t* tile, uint32_t* tiles_x, uint32_t* tiles_y, uint64_t* capacity)
{
    if (!h || !tile || !tiles_x || !tiles_y || !capacity) return SSIMU2_E_INVALID;
    *tile = h->tile;
    *tiles_x = h->tiles_x;
    *tiles_y = h->tiles_y;
    *capacity = h->tile_cap;
    return SSIMU2_OK;
}

int ssimu2_get_tile_scores(ssimu2_t* h, uint64_t ticket, double* out, size_t n)
{
    if (!h || !out) return SSIMU2_E_INVALID;
    if (!h->tile) return SSIMU2_E_UNSUPPORTED;
    const size_t nt = (size_t)h->tiles_x * h->tiles_y;
    if (n < nt) return SSIMU2_E_INVALID;
    if (ticket >= h->next_ticket || h->next_ticket - ticket > h->tile_cap) return SSIMU2_E_TICKET;
    int r = ssimu2_wait(h, ticket);
    if (r) return r;
    memcpy(out, &h->res_tiles[(ticket % h->tile_cap) * nt], nt * sizeof(double));
    return SSIMU2_OK;
}

int ssimu2_scores_device(ssimu2_t* h, uint64_t* dptr, uint64_t* capacity)
{
    if (!h || !dptr || !capacity) return SSIMU2_E_INVALID;
    *dptr = (uint64_t)(uintptr_t)h->scores_ring_d;
    *capacity = kResultCap;
    return SSIMU2_OK;
}

int ssimu2_get_info(const ssimu2_t* h, ssimu2_info* info)
{
    if (!h || !info) return SSIMU2_E_INVALID;
    memset(info, 0, sizeof(*info));
    info->nscales = (uint32_t)h->geo.nscales;
    for (int s = 0; s < h->geo.nscales; s++) {
        info->width[s] = (uint32_t)h->geo.sc[s].w;
        info->height[s] = (uint32_t)h->geo.sc[s].h;
        info->pitch[s] = (uint32_t)h->geo.sc[s].pitch;
    }
    info->batch = h->batch;
    info->ring = h->ring;
    info->alg_bytes_per_pair = h->alg_bytes;
    info->kernel_launches = h->launches;
    info->pipeline = (uint32_t)h->pipeline;
    info->flags = h->cfg.flags;
    info->input_group = h->input_group;
    info->strips_per_pair = (uint32_t)h->geo.items_v;
    info->io_bytes_per_pair = h->io_bytes;
    return SSIMU2_OK;
}

// ---- include/ssimu2_b200_debug.h ---------------------------------------------------------------
// The batch slot that served `ticket` and the ticket's frame index in it (valid until the slot is reused).
static int debug_slot(ssimu2_t* h, uint64_t ticket, Slot** sl, size_t* idx)
{
    int si = h->res_slot[ticket % kResultCap];
    if (si < 0) return SSIMU2_E_TICKET;
    *sl = &h->slots[si];
    if (ticket < (*sl)->first_ticket) return SSIMU2_E_TICKET;
    *idx = (size_t)(ticket - (*sl)->first_ticket);
    if (*idx >= h->batch) return SSIMU2_E_TICKET;
    return SSIMU2_OK;
}

int ssimu2_debug_read(ssimu2_t* h, uint64_t ticket, int what, int scale, float* out, size_t out_floats)
{
    if (!h || !out || scale < 0 || scale >= h->geo.nscales) return SSIMU2_E_INVALID;
    int r = ssimu2_wait(h, ticket);
    if (r) return r;
    DeviceGuard guard(h->cfg.device);
    Slot* slp;
    size_t idx;
    if ((r = debug_slot(h, ticket, &slp, &idx))) return r;
    Slot& sl = *slp;
    const ScaleDesc& sd = h->geo.sc[scale];
    int planes;
    const float* src;
    if (what == 0) {
        planes = 6;
        src = sl.xyb + idx * h->geo.xyb_stride + sd.xyb_off;
    } else if (what == 1) {
        if (!sl.hb) return SSIMU2_E_UNSUPPORTED;  // the fused H+V pipeline never materialises these planes
        planes = 15;
        src = sl.hb + idx * h->geo.hb_stride + sd.hb_off;
    } else {
        return SSIMU2_E_INVALID;
    }
    if (out_floats < (size_t)planes * sd.w * sd.h) return SSIMU2_E_INVALID;
    CU_TRY(cudaMemcpy2D(out, (size_t)sd.w * sizeof(float), src, (size_t)sd.pitch * sizeof(float),
                        (size_t)sd.w * sizeof(float), (size_t)planes * sd.h, cudaMemcpyDeviceToHost));
    return SSIMU2_OK;
}

int ssimu2_debug_read_partials(ssimu2_t* h, uint64_t ticket, double* out, size_t out_doubles)
{
    if (!h || !out) return SSIMU2_E_INVALID;
    int r = ssimu2_wait(h, ticket);
    if (r) return r;
    DeviceGuard guard(h->cfg.device);
    Slot* sl;
    size_t idx;
    if ((r = debug_slot(h, ticket, &sl, &idx))) return r;
    const size_t n = (size_t)h->geo.total_strips * 18;
    if (out_doubles < n) return SSIMU2_E_INVALID;
    CU_TRY(cudaMemcpy(out, sl->partials + idx * n, n * sizeof(double), cudaMemcpyDeviceToHost));
    return SSIMU2_OK;
}

int ssimu2_debug_strips(const ssimu2_t* h, uint32_t strip0[6], uint32_t n_strips[6], uint32_t* strip_cols)
{
    if (!h || !strip0 || !n_strips || !strip_cols) return SSIMU2_E_INVALID;
    for (int s = 0; s < kMaxScales; s++) {
        const bool on = s < h->geo.nscales;
        strip0[s] = on ? (uint32_t)h->geo.sc[s].strip0 : 0u;
        n_strips[s] = on ? (uint32_t)h->geo.sc[s].n_strips : 0u;
    }
    *strip_cols = (uint32_t)kVCols;
    return SSIMU2_OK;
}

int ssimu2_debug_read_tile_partials(ssimu2_t* h, uint64_t ticket, double* out, size_t out_doubles)
{
    if (!h || !out) return SSIMU2_E_INVALID;
    if (!h->tile) return SSIMU2_E_UNSUPPORTED;
    int r = ssimu2_wait(h, ticket);
    if (r) return r;
    DeviceGuard guard(h->cfg.device);
    Slot* sl;
    size_t idx;
    if ((r = debug_slot(h, ticket, &sl, &idx))) return r;
    const size_t n = h->tile_entries * 18;
    if (out_doubles < n) return SSIMU2_E_INVALID;
    CU_TRY(cudaMemcpy(out, sl->tiles + idx * n, n * sizeof(double), cudaMemcpyDeviceToHost));
    return SSIMU2_OK;
}

int ssimu2_debug_tile_units(const ssimu2_t* h, uint32_t entry0[6], uint32_t units[6], uint32_t unit_cols[6])
{
    if (!h || !entry0 || !units || !unit_cols) return SSIMU2_E_INVALID;
    if (!h->tile) return SSIMU2_E_UNSUPPORTED;
    for (int s = 0; s < kMaxScales; s++) {
        int u = 0;
        const bool on = s < h->geo.nscales;
        entry0[s] = on ? (uint32_t)tile_layout(h->geo, h->tile_log2, s, &u) : 0u;
        units[s] = on ? (uint32_t)u : 0u;
        unit_cols[s] = on ? std::min<uint32_t>(64u, h->tile >> s) : 0u;
    }
    return SSIMU2_OK;
}

#ifdef KX_TRACE
extern "C" int ssimu2_debug_hv_trace(unsigned long long* out)
{
    return (int)cudaMemcpyFromSymbol(out, ssimu2::g_hv_trace, sizeof(ssimu2::g_hv_trace));
}
#endif
int ssimu2_debug_math(int op, const float* in, float y, float* out, size_t n)
{
    if (!in || !out || op < 0 || op > 6) return SSIMU2_E_INVALID;
    if (n == 0) return SSIMU2_OK;
    const size_t in_b = op == 3 ? n * 16 : (op == 4 ? n * 8 : n * 4), out_b = op == 3 ? n * 8 : n * 4;
    float *din = nullptr, *dout = nullptr;
    if (cudaMalloc(&din, in_b) != cudaSuccess || cudaMalloc(&dout, out_b) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(din);
        return SSIMU2_E_NOMEM;
    }
    int rc = (int)cudaMemcpy(din, in, in_b, cudaMemcpyHostToDevice);
    if (!rc) {
        k_debug_math<<<(unsigned)((n + 255) / 256), 256>>>(op, din, y, dout, n);
        rc = (int)cudaGetLastError();
    }
    if (!rc) rc = (int)cudaMemcpy(out, dout, out_b, cudaMemcpyDeviceToHost);
    cudaFree(din);
    cudaFree(dout);
    return rc;
}

int ssimu2_last_batch_ms(ssimu2_t* h, float ms[4])
{
    if (!h || !ms) return SSIMU2_E_INVALID;
    memcpy(ms, h->last_ms, sizeof(h->last_ms));
    return SSIMU2_OK;
}

int ssimu2_kernel_ms(ssimu2_t* h, double ms_total[4], uint64_t* batches, uint64_t* pairs, int reset)
{
    if (!h || !ms_total) return SSIMU2_E_INVALID;
    for (int k = 0; k < 4; k++) ms_total[k] = h->total_ms[k];
    if (batches) *batches = h->timed_batches;
    if (pairs) *pairs = h->timed_pairs;
    if (reset) {
        for (int k = 0; k < 4; k++) h->total_ms[k] = 0;
        h->timed_batches = h->timed_pairs = 0;
    }
    return SSIMU2_OK;
}

}  // extern "C"
