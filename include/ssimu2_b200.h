/*
 * ssimu2_b200.h -- C ABI of the B200-native SSIMULACRA2 frame-pair scorer.
 *
 * Drop-in boundary for the reference's `Ssimulacra2` metric op and the colour front-end
 * that feeds it (paths relative to /root/reference/crates):
 *
 *   ssimulacra2-cuda/src/lib.rs:27-107   struct Ssimulacra2 / Ssimulacra2::new      -> ssimu2_create
 *   turbo-metrics/src/lib.rs:268-360     compute_one(fref, cc_ref, fdis, cc_dis)    -> ssimu2_create_mixed when the two
 *                                        sources differ in HwFrame variant or colour characteristics
 *   ssimulacra2-cuda/src/lib.rs:110      Ssimulacra2::mem_usage                     -> ssimu2_mem_usage
 *   ssimulacra2-cuda/src/lib.rs:283-287  Ssimulacra2::compute (async)               -> ssimu2_submit
 *   ssimulacra2-cuda/src/lib.rs:271-279  Ssimulacra2::compute_sync                  -> ssimu2_compute_sync
 *   ssimulacra2-cuda/src/lib.rs:253-266  Ssimulacra2::compute_srgb_sync             -> ssimu2_compute_sync (SSIMU2_FMT_SRGB8)
 *   ssimulacra2-cuda/src/lib.rs:232-250  Ssimulacra2::compute_from_cpu_srgb_sync    -> ssimu2_submit_host + ssimu2_get_score
 *   ssimulacra2-cuda/src/lib.rs:289-291  Ssimulacra2::get_score                     -> ssimu2_get_score
 *   cudarse-video/src/dec.rs:277-287     FrameMapping drop (surface reuse)          -> ssimu2_stream_wait_input
 *   cuda-colorspace/src/lib.rs:33-123    ColorspaceConversion::biplanaryuv420_to_linearrgb_{8,16}
 *                                        (folded into the scorer: SSIMU2_FMT_NV12 / SSIMU2_FMT_P016)
 *   cuda-colorspace/src/lib.rs:144-169   srgb_to_linear_{u8,u16,f32}                (SSIMU2_FMT_SRGB8/16/F32)
 *   turbo-metrics/src/lib.rs:268-360     TurboMetrics::compute_one (the caller)     -> ssimu2_submit / ssimu2_get_score
 *   turbo-metrics/src/lib.rs:362-433     TurboMetrics::compute_all frame loop       -> ssimu2_submit_batch + tickets;
 *                                        across the GPUs of a box                   -> ssimu2_shard_*
 *
 * Conventions
 *   - Plain C types only.  Device pointers are CUdeviceptr-compatible 64-bit integers,
 *     streams are CUstream / cudaStream_t handles passed as void*.
 *   - Every function returns 0 (SSIMU2_OK) or a negative ssimu2_status; a positive value is
 *     a CUDA runtime error code passed through.  Nothing throws or aborts across the ABI.
 *   - Input frames are BORROWED: read-only, never freed.  LIFETIME RULE: the scorer reads a frame when its batch (or,
 *     with cfg.input_group, its input group) is LAUNCHED, which can be later than ssimu2_submit returns.  A frame must
 *     therefore stay valid AND UNMODIFIED until one of: ssimu2_wait / ssimu2_get_score / ssimu2_get_scores has
 *     returned for its ticket; ssimu2_completed reports a watermark above its ticket; or the stream that will
 *     overwrite it has been made to wait with ssimu2_stream_wait_input (inputs consumed) or ssimu2_stream_wait (batch
 *     done).  The reference enqueues its graph on the caller's stream at once and syncs per pair
 *     (turbo-metrics/src/lib.rs:342-358); here the dependency on the caller's stream is recorded at submit time, so
 *     everything enqueued on `stream` BEFORE the submit is seen, and nothing enqueued after it is waited for.
 *   - Decoder-style surface pools (cudarse-video/src/dec.rs:277-287: a surface is valid until unmapped): set
 *     cfg.input_group (pairs per front-end launch, e.g. 1-4) so that surfaces are consumed shortly after submit, and
 *     recycle each one behind ssimu2_stream_wait_input(ticket, decoder_stream) -- no host synchronisation.
 *   - Scales: like the reference's CPU implementation (cpu.rs:359) a frame whose scale-s size is below 8x8 stops the
 *     pyramid at s+1 scales (fewer than 6 for min(width, height) < 113) and the 108 weights are consumed densely over
 *     the scales that exist.  The reference's GPU op always runs 6 scales with fixed weight offsets
 *     (ssimulacra2-cuda/src/lib.rs:61-65, 586-603) and gives a different score for such small frames; the parity
 *     target named by BASELINE.json is the CPU implementation.  ssimu2_info.nscales tells which case applies.
 *   - A handle is bound to one device and one (width, height, format).  Calls on one handle
 *     are not re-entrant; different handles may be driven from different threads.
 *   - Mixed sources: ssimu2_create_mixed binds the distorted frames to a description of their own (format, matrix, range),
 *     like TurboMetrics::compute_one(fref, cc_ref, fdis, cc_dis), which converts each frame with its own HwFrame variant and
 *     colour characteristics (turbo-metrics/src/lib.rs:268-360).  The distorted frames may also be smaller than the
 *     reference (ssimu2_source.width / height: an encoding ladder's lower rungs against their source); they are upscaled
 *     to the reference's size on the GPU with a fixed bicubic filter before they are scored (see ssimu2_source).
 *   - There is no CPU fallback: if no CUDA device is usable every entry point fails.
 */
#ifndef SSIMU2_B200_H
#define SSIMU2_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ssimu2_handle ssimu2_t;

typedef enum {
    SSIMU2_OK = 0,
    SSIMU2_E_INVALID = -1,     /* bad argument */
    SSIMU2_E_UNSUPPORTED = -2, /* format / size not supported (reference: todo!() panics) */
    SSIMU2_E_NOMEM = -3,
    SSIMU2_E_NODEVICE = -4, /* no CUDA device / not an sm_100 part */
    SSIMU2_E_TICKET = -5,   /* ticket unknown or already overwritten in the result ring */
    SSIMU2_E_INTERNAL = -6
} ssimu2_status;

/* Pixel formats crossing the boundary (turbo-metrics/src/lib.rs:125-130 `HwFrame`). */
typedef enum {
    SSIMU2_FMT_NV12 = 0,      /* NvDecFrame::NV12: u8 Y plane + interleaved u8 CbCr plane, 4:2:0 */
    SSIMU2_FMT_P016 = 1,      /* NvDecFrame::P016: u16 MSB-aligned Y + interleaved CbCr, 4:2:0 */
    SSIMU2_FMT_SRGB8 = 2,     /* Npp8 : packed RGB u8, sRGB transfer (256-entry table) */
    SSIMU2_FMT_SRGB16 = 3,    /* Npp16: packed RGB u16, sRGB transfer (analytic) */
    SSIMU2_FMT_SRGBF32 = 4,   /* Npp32: packed RGB f32 in [0,1], sRGB transfer (analytic) */
    SSIMU2_FMT_LINEARF32 = 5, /* packed linear RGB f32: the input of Ssimulacra2::new itself */
    /* ABI 2.3: NVDEC's 4:2:2 and 4:4:4 surfaces (cudaVideoSurfaceFormat_NV16 / _P216 / _YUV444 / _YUV444_16Bit).  Chroma is
     * sited nearest-neighbour, like the 4:2:0 formats: pixel (x, y) takes chroma (x >> 1, y) in 4:2:2, (x, y) in 4:4:4. */
    SSIMU2_FMT_NV16 = 8,      /* u8 Y plane + interleaved u8 CbCr plane of full height, 4:2:2 */
    SSIMU2_FMT_P216 = 9,      /* u16 MSB-aligned Y + interleaved CbCr of full height, 4:2:2 */
    SSIMU2_FMT_YUV444 = 10,   /* u8 Y, Cb and Cr planes, 4:4:4 */
    SSIMU2_FMT_YUV444P16 = 11 /* u16 MSB-aligned Y, Cb and Cr planes, 4:4:4 */
} ssimu2_format;

/* cuda-colorspace/src/lib.rs:8-13 `ColorMatrix` (only used by the YUV formats). */
typedef enum { SSIMU2_MATRIX_BT709 = 0, SSIMU2_MATRIX_BT601_525 = 1, SSIMU2_MATRIX_BT601_625 = 2 } ssimu2_matrix;

/* One device frame.  YUV 4:2:0: plane[0] = Y, plane[1] = interleaved CbCr, ceil(height / 2) rows
 * (NVDEC: plane[1] = plane[0] + pitch * coded_height, cudarse-video/src/dec.rs:299-366, but any placement works: a separate
 * allocation, chroma before luma, coded_height == height), both with the same pitch.  YUV 4:2:2 (NV16, P216): the same with
 * `height` rows of interleaved CbCr.  YUV 4:4:4 (YUV444, YUV444P16): plane[1] = Cb, and the Cr plane lies at
 * plane[1] + (plane[1] - plane[0]), all three with the same pitch -- NVDEC's layout (planes pitch x coded_height apart) and that of
 * a contiguous (3, H, pitch) array; ssimu2_frame has no third address.  Packed RGB formats use plane[0] only.
 * Layout rule (SSIMU2_E_INVALID otherwise, ABI 2.2; 4:2:2 and 4:4:4 since 2.3):
 *   - pitch is in bytes and holds one row: width x 3 / 6 / 12 bytes for sRGB8 / sRGB16 / the f32 formats; for NV12 / P016 /
 *     NV16 / P216 width luma samples and 2 x ceil(width / 2) chroma samples, for YUV444 / YUV444P16 width samples (1 / 2 bytes
 *     each);
 *   - everything is aligned to one sample (1 byte: NV12, NV16, YUV444, sRGB8; 2: P016, P216, YUV444P16, sRGB16; 4: sRGB f32,
 *     linear f32): for device frames plane[0], plane[1] and pitch (4:4:4: the Cr address must not wrap around the address space);
 *     for host frames pitch and plane[1] - plane[0] (host frames are staged to aligned memory);
 *   - host frames: the byte count copied from plane[0] covers (height - 1) x pitch + the row bytes and, for YUV, the end of the
 *     last chroma row: (plane[1] - plane[0]) + (ceil(height / 2) - 1) x pitch + the chroma row bytes for 4:2:0,
 *     (plane[1] - plane[0]) + (height - 1) x pitch + the chroma row bytes for 4:2:2, 2 x (plane[1] - plane[0]) + (height - 1) x
 *     pitch + the row bytes for 4:4:4 (the last Cr row).
 * Rows may be padded and may lie more than 4 GiB past plane[0].  The batch entry points (ssimu2_submit_batch,
 * ssimu2_submit_host_batch / _sized, ssimu2_shard_submit_*) check every pair before queueing any: on SSIMU2_E_INVALID nothing of
 * the call was accepted. */
typedef struct {
    uint64_t plane[2];
    uint32_t pitch;
    uint32_t reserved;
} ssimu2_frame;

typedef enum {
    SSIMU2_PIPELINE_DEFAULT = 0, /* front-end, fused H+V filter/map/sum kernel, finalize */
    SSIMU2_PIPELINE_SPLIT = 1    /* development: separate H and V passes, H-pass planes kept in HBM (ssimu2_debug_read) */
} ssimu2_pipeline;

/* ssimu2_config.flags */
#define SSIMU2_FLAG_SCORE_ONLY 1u /* compute only what the score depends on: the filters and SSIM map of every (scale, channel) \
                                     whose two SSIM weights are both zero are skipped (the reference computes them and multiplies \
                                     by 0.0, ssimulacra2-cuda/src/lib.rs:586-603).  Scores are bit-identical to the full mode;    \
                                     ssimu2_get_norms returns SSIMU2_E_UNSUPPORTED. */
#define SSIMU2_FLAG_NO_TIMING 2u  /* do not record the per-kernel timing events (ssimu2_b200_debug.h) */
#define SSIMU2_FLAG_P016_DEEP 4u  /* SSIMU2_FMT_P016, _P216 and _YUV444P16 only: the samples carry more than 10 significant bits \
                                     (12-bit sources, e.g. HEVC Main12 / Main 4:4:4 12 through NVDEC).  Results never depend on this flag; it selects a front-end that      \
                                     evaluates all three transfer functions instead of the exact 10-bit memo tables, which such  \
                                     content cannot use (without the flag it is scored correctly, at a third of the speed). */

typedef struct {
    uint32_t width, height;
    int32_t format;       /* ssimu2_format */
    int32_t matrix;       /* ssimu2_matrix */
    int32_t full_range;   /* 0 = limited (what the reference implements), 1 = full */
    int32_t device;       /* CUDA device ordinal */
    uint32_t batch;       /* frame pairs per kernel launch group, at most 1024.  0 = chosen from the frame size: 8 at 4K, 32 at
                             1080p, 128 for 512x512 (enough strips for ~8 waves, workspace of all ring slots <= 8 GiB) */
    uint32_t ring;        /* batches in flight, one stream each (0 = default 3) */
    uint32_t pipeline;    /* ssimu2_pipeline */
    uint32_t flags;       /* SSIMU2_FLAG_* */
    uint32_t input_group; /* pairs per front-end launch; 0 = whole batch.  Smaller groups consume the input frames sooner */
    uint32_t tile;        /* tile scores (see below); 0 = off */
    uint32_t reserved[4]; /* must be 0 */
} ssimu2_config;

/* Tile scores (ssimu2_config.tile, since ABI 2.3; ssimu2_version() is unchanged, so probe the capability by creating a handle:
 * an older library returns SSIMU2_E_INVALID for the word).  Besides its frame score, every pair gets a coarse map: one
 * SSIMULACRA2 score per tile of a grid, for finding WHERE a frame is bad.
 *   - tile = T, a power of two with 64 <= T <= 32768 (otherwise SSIMU2_E_UNSUPPORTED, as is any T with SSIMU2_PIPELINE_SPLIT;
 *     both checked before any device call; ssimu2_shard_create / _create_mixed refuse any T != 0).  Tile (ty, tx) covers
 *     the pixels [tx T, (tx + 1) T) x [ty T, (ty + 1) T), clipped to the frame: tiles_x = ceil(width / T) by
 *     tiles_y = ceil(height / T) tiles.
 *   - The pyramid nests exactly: scale-s pixel i is the box of scale-0 pixels [i 2^s, (i + 1) 2^s).  At scale s a tile's
 *     footprint is the T_s = T >> s square at (tx T_s, ty T_s), clipped to that scale's size; it is never empty.
 *   - The maps are those of the frame score, computed over the whole frame; only the pooling is restricted.  Per tile, scale
 *     s, channel c and map m: L1 = sum over the footprint of the map / N_s and L4 = (sum of map^4 / N_s)^(1/4), N_s the
 *     footprint's pixel count.  These 108 norms (WEIGHT order, see ssimu2_get_norms) give the score exactly as the frame's
 *     norms give the frame score: the dense weight cursor over the scales that exist, x 0.9562..., the cubic, and
 *     100 - 10 s^0.6276... (s <= 0 gives 100).
 *   - So a tile score is NOT the score of the cropped tile (a crop would zero-pad the filters at its edges), the frame score
 *     is NOT the mean of the tile scores, and a tile whose reference and distorted neighbourhoods are identical scores
 *     exactly 100.  Frame scores and norms are bit-identical to those of the same handle without tiles, and tile scores are
 *     bit-identical between the full and the score-only mode. */

/* The description of the DISTORTED frames of a mixed handle (ssimu2_create_mixed); ssimu2_config describes the reference. */
typedef struct {
    int32_t format;       /* ssimu2_format of the distorted frames */
    int32_t matrix;       /* ssimu2_matrix (YUV formats) */
    int32_t full_range;   /* 0 = limited, 1 = full */
    uint32_t flags;       /* SSIMU2_FLAG_P016_DEEP only, and only with a 16-bit YUV format (P016, P216, YUV444P16) */
    /* Scaled distorted frames: the size of the distorted frames, 1 <= width <= cfg.width and 1 <= height <= cfg.height
     * (a larger side is SSIMU2_E_UNSUPPORTED, one of the two 0 is SSIMU2_E_INVALID).  0, 0 = the reference's size.  The pair is
     * scored at the reference's size: each distorted frame is first upscaled in its own sample domain to a frame of the same
     * format at cfg.width x cfg.height, plane by plane on the plane's own grid (4:2:0 chroma ceil(width / 2) x ceil(height / 2)
     * -> ceil(cfg.width / 2) x ceil(cfg.height / 2); 4:2:2 chroma ceil(width / 2) x height -> ceil(cfg.width / 2) x cfg.height;
     * 4:4:4 chroma and packed RGB as luma; interleaved Cb / Cr and the three RGB channels each on their own).  The filter is
     * separable bicubic Catmull-Rom (Keys, a = -0.5), centre-aligned (sx = (x + 0.5) * in / out - 0.5), clamp-to-edge, taps
     * floor(sx) - 1 .. floor(sx) + 2, weights computed in double and rounded to float, evaluated in f32 horizontally first as
     * a = w0 * s0 followed by three fmaf steps.  u8 / u16 results are rounded half to even and clamped to [0, 255] /
     * [0, 65535] (16-bit results are not re-quantised to 10 bits); f32 results are stored unrounded and unclamped.  An axis
     * whose size is unchanged is copied exactly.  This is NOT ffmpeg swscale's bicubic (B = 0, C = 0.6, fixed point): scores
     * differ from those of an ffmpeg-upscaled pipeline by that difference.  Since ABI 2.3; ssimu2_version() is unchanged, so
     * probe the capability by creating a handle: an older library returns SSIMU2_E_INVALID for these words.  Distorted frames
     * are checked against the layout rule at their own size (host byte counts too). */
    uint32_t width, height;
    uint32_t reserved[2]; /* must be 0 */
} ssimu2_source;

/* ---- lifetime ------------------------------------------------------------------------ */
int ssimu2_create(ssimu2_t **out, const ssimu2_config *cfg);
/* A handle whose distorted frames have their own pixel format / matrix / range.  cfg describes the reference frames (its
 * SSIMU2_FLAG_P016_DEEP applies to the reference side only); dis == NULL: exactly ssimu2_create.  `dis` is checked before any
 * device call: a bad format or matrix, a flag other than SSIMU2_FLAG_P016_DEEP, or that flag with a format other than P016 / P216
 * / YUV444P16 is SSIMU2_E_UNSUPPORTED; non-zero reserved fields are SSIMU2_E_INVALID.  When the two sides are the same effective description
 * (same format and deep flag; for the YUV formats also the same matrix and range; the same size) the result is an ordinary handle: one
 * front-end launch per input group and the same bits.  Otherwise the front-end runs once per side on the slot's stream, and
 * the frames of each side are checked against that side's format and size (ssimu2_frame pitch rule).  A scaled handle runs
 * three kernels per input group: the reference's front-end, the upscale of the distorted frames into handle-owned staging
 * memory (one frame of the distorted format at the reference's size per pair of an input group, per ring slot) and the
 * distorted side's front-end.  Its io / alg bytes per pair count the distorted input at its own size. */
int ssimu2_create_mixed(ssimu2_t **out, const ssimu2_config *cfg, const ssimu2_source *dis);
int ssimu2_destroy(ssimu2_t *h);
/* Device bytes owned by the handle (Ssimulacra2::mem_usage). */
int ssimu2_mem_usage(const ssimu2_t *h, size_t *bytes);
const char *ssimu2_strerror(int status);
/* Library / ABI version: (major << 16) | minor. */
uint32_t ssimu2_version(void);

/* ---- scoring: device frames ---------------------------------------------------------- */
/* Enqueue one pair.  Work is ordered after everything already enqueued on `stream` (may be
 * NULL = legacy default stream).  Never blocks on the GPU unless the ring is full.  Pairs are
 * grouped into batches of cfg.batch; a partial batch is launched by ssimu2_flush or by
 * fetching one of its tickets.  Tickets increase by 1 per pair in submission order. */
int ssimu2_submit(ssimu2_t *h, const ssimu2_frame *ref, const ssimu2_frame *dis, void *stream, uint64_t *ticket);
/* n pairs at once; *first_ticket receives the ticket of pair 0 (pair i has first_ticket+i). */
int ssimu2_submit_batch(ssimu2_t *h, uint32_t n, const ssimu2_frame *refs, const ssimu2_frame *diss, void *stream,
                        uint64_t *first_ticket);
/* Launch whatever is pending. */
int ssimu2_flush(ssimu2_t *h);
/* Block until the ticket's batch has completed on the device. */
int ssimu2_wait(ssimu2_t *h, uint64_t ticket);
/* *watermark = the lowest ticket whose results have not reached the host yet: every pair below it has completed and its
 * input frames are no longer referenced (batches complete out of order across ring slots; this is the in-order bound). */
int ssimu2_completed(ssimu2_t *h, uint64_t *watermark);
/* Score of a ticket (flushes and waits as needed).  100 = identical, unbounded below. */
int ssimu2_get_score(ssimu2_t *h, uint64_t ticket, double *score);
/* The scores of n consecutive tickets in submission order: the per-frame score stream of the CLI loop
 * (turbo-metrics-cli/src/main.rs:307-322) in one call. */
int ssimu2_get_scores(ssimu2_t *h, uint64_t first_ticket, uint32_t n, double *scores);
/* The 108 per-scale / per-channel norms in WEIGHT order:
 * index = channel*36 + scale*6 + norm*3 + map, norm in {L1,L4}, map in {ssim, artifact, detail}. */
int ssimu2_get_norms(ssimu2_t *h, uint64_t ticket, double *norms108);
/* Submit + wait + score in one call (Ssimulacra2::compute_sync). */
int ssimu2_compute_sync(ssimu2_t *h, const ssimu2_frame *ref, const ssimu2_frame *dis, void *stream, double *score);
/* Make `stream` wait (device side) until the ticket's batch is done, so the caller may
 * recycle the input frames in stream order without a host sync. */
int ssimu2_stream_wait(ssimu2_t *h, uint64_t ticket, void *stream);
/* Same, but only until the ticket's INPUT FRAMES have been consumed (its front-end launch is done); launches the pending
 * input group if the ticket is still waiting in one.  This is the call that lets a decoder reuse a surface. */
int ssimu2_stream_wait_input(ssimu2_t *h, uint64_t ticket, void *stream);

/* ---- scoring: host frames ------------------------------------------------------------ */
/* Ssimulacra2::compute_from_cpu_srgb_sync generalised to every format: the frames live in
 * HOST memory with the same layout an ssimu2_frame describes (plane[] are host addresses;
 * for YUV plane[1] must lie inside the same allocation as plane[0], after it).  The library
 * copies them to its own device staging ring (pinned memory is faster but not required) and
 * enqueues the pair.  frame_bytes = bytes to copy starting at plane[0].
 * Lifetime: a PAGEABLE buffer has been read when the call returns (the CUDA runtime stages it) and may be reused at once,
 * like the slices of the reference's call; a PINNED buffer is read asynchronously by the copy engine: keep it unmodified
 * until the pair's score has been fetched or ssimu2_completed() has passed its ticket. */
int ssimu2_submit_host(ssimu2_t *h, const ssimu2_frame *ref, const ssimu2_frame *dis, size_t frame_bytes,
                       uint64_t *ticket);
/* n host pairs at once (all frames share frame_bytes); pair i has *first_ticket + i.  The frame loop of a caller that
 * decodes on the CPU (turbo-metrics/src/input_image.rs:206-228 copies each frame itself) becomes one call per chunk. */
int ssimu2_submit_host_batch(ssimu2_t *h, uint32_t n, const ssimu2_frame *refs, const ssimu2_frame *diss,
                             size_t frame_bytes, uint64_t *first_ticket);
/* Host frames whose two sides have different sizes (a mixed handle, e.g. an NV12 reference against a P016 encode): reference i
 * copies ref_bytes starting at refs[i].plane[0], distorted i copies dis_bytes.  Otherwise as ssimu2_submit_host_batch, which
 * (like ssimu2_submit_host) is this call with ref_bytes == dis_bytes and returns SSIMU2_E_INVALID on a mixed handle whose
 * two sides have different bytes per pixel. */
int ssimu2_submit_host_sized(ssimu2_t *h, uint32_t n, const ssimu2_frame *refs, size_t ref_bytes, const ssimu2_frame *diss,
                             size_t dis_bytes, uint64_t *first_ticket);

/* ---- tile scores (ssimu2_config.tile) ------------------------------------------------------ */
/* The handle's tile grid: *tile = ssimu2_config.tile (0: a handle without tiles, the rest 0 too), tiles_x x tiles_y tiles, and
 * *capacity = how many of the most recent tickets still have their map on the host (at least batch x ring). */
int ssimu2_get_tile_grid(const ssimu2_t *h, uint32_t *tile, uint32_t *tiles_x, uint32_t *tiles_y, uint64_t *capacity);
/* The tile scores of a ticket: tiles_y x tiles_x doubles, row-major (flushes and waits like ssimu2_get_score).
 * SSIMU2_E_UNSUPPORTED on a handle without tiles, SSIMU2_E_INVALID if n is smaller than tiles_x x tiles_y, SSIMU2_E_TICKET
 * for a ticket not submitted yet or older than the capacity. */
int ssimu2_get_tile_scores(ssimu2_t *h, uint64_t ticket, double *out, size_t n);

/* ---- results on the device ----------------------------------------------------------- */
/* Device address of the f64 score ring (one entry per ticket, index ticket % capacity). */
int ssimu2_scores_device(ssimu2_t *h, uint64_t *dptr, uint64_t *capacity);

/* ---- introspection ----------------------------------------------------------------- */
typedef struct {
    uint32_t nscales;
    uint32_t width[6], height[6], pitch[6]; /* pitch in floats */
    uint32_t batch, ring;
    uint64_t alg_bytes_per_pair; /* B_alg of SURVEY.md section 8(d) for this geometry */
    uint64_t kernel_launches;    /* kernels launched so far by this handle */
    uint32_t pipeline, flags, input_group;
    uint32_t strips_per_pair;    /* k_hv work items (64-column strips over all scales) per pair */
    uint64_t io_bytes_per_pair;  /* B_io: compulsory input bytes of a pair + 8 (SURVEY.md section 8d) */
} ssimu2_info;
int ssimu2_get_info(const ssimu2_t *h, ssimu2_info *info);

/* ---- frame-sharded scoring across the GPUs of one box (ssimu2_shard.cu) -------------------------------------------
 * The reference drives one GPU (device 0 is hard-coded, turbo-metrics/src/lib.rs:438-456) from one thread
 * (frame loop turbo-metrics/src/lib.rs:362-433).  SSIMULACRA2 pairs are independent (ssimulacra2-cuda/README.md:26-27),
 * so N GPUs = N handles, each driven by its own host thread INSIDE the library; the caller keeps the single-threaded
 * submit / fetch loop.  Global tickets increase by one per pair in submission order; pair g goes to device
 * (g / cfg.batch) % n_devices (whole batches stay on one GPU).  No collective, no peer access: only f64 scores leave a GPU.
 * Frames are HOST frames (any device would need them anyway): each worker copies its pairs to its own GPU. */
typedef struct ssimu2_shard ssimu2_shard_t;
/* cfg->device is ignored; devices[i] are CUDA ordinals (n_devices >= 1). */
int ssimu2_shard_create(ssimu2_shard_t **out, const ssimu2_config *cfg, const int32_t *devices, uint32_t n_devices);
/* Every worker's handle is ssimu2_create_mixed(cfg, dis); dis == NULL: ssimu2_shard_create. */
int ssimu2_shard_create_mixed(ssimu2_shard_t **out, const ssimu2_config *cfg, const ssimu2_source *dis, const int32_t *devices,
                              uint32_t n_devices);
int ssimu2_shard_destroy(ssimu2_shard_t *s);
/* n host pairs (layout as ssimu2_submit_host); returns at once, the copies and launches run on the worker threads.
 * The frames must stay valid until their scores have been fetched.  *first_ticket = global ticket of pair 0. */
int ssimu2_shard_submit_host(ssimu2_shard_t *s, uint32_t n, const ssimu2_frame *refs, const ssimu2_frame *diss,
                             size_t frame_bytes, uint64_t *first_ticket);
/* Host pairs with one byte count per side (layout as ssimu2_submit_host_sized); otherwise as ssimu2_shard_submit_host. */
int ssimu2_shard_submit_host_sized(ssimu2_shard_t *s, uint32_t n, const ssimu2_frame *refs, size_t ref_bytes,
                                   const ssimu2_frame *diss, size_t dis_bytes, uint64_t *first_ticket);
/* n DEVICE pairs that already live on the GPU the sharding rule assigns them to (ssimu2_shard_device_of); `streams[d]`
 * (may be NULL = no dependency) is the stream of device d the frames were produced on. */
int ssimu2_shard_submit_device(ssimu2_shard_t *s, uint32_t n, const ssimu2_frame *refs, const ssimu2_frame *diss,
                               void *const *streams, uint64_t *first_ticket);
/* CUDA ordinal that global ticket `ticket` is (or will be) scored on. */
int ssimu2_shard_device_of(const ssimu2_shard_t *s, uint64_t ticket, int32_t *device);
/* Scores of n consecutive global tickets, in submission order (blocks until they are done). */
int ssimu2_shard_get_scores(ssimu2_shard_t *s, uint64_t first_ticket, uint32_t n, double *scores);
int ssimu2_shard_flush(ssimu2_shard_t *s);

#ifdef __cplusplus
}
#endif
#endif /* SSIMU2_B200_H */
