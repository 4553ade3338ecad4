/*
 * ssimu2_b200_debug.h -- test / measurement hooks of libssimu2_b200.so.  NOT part of the drop-in boundary
 * (include/ssimu2_b200.h): the parity tests read intermediate planes and run the device arithmetic helpers through
 * these, bench.py reads the per-kernel CUDA-event times.
 */
#ifndef SSIMU2_B200_DEBUG_H
#define SSIMU2_B200_DEBUG_H

#include "ssimu2_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Copy an intermediate plane set of the batch slot that served `ticket` to host memory.
 * what = 0: XYB planes of `scale`:                float[2][3][h][w]  (ref X,Y,B then dis X,Y,B)
 * what = 1: H-pass output of `scale`:            float[15][h][w]    (s11,s22,s12,mu1,mu2) x 3 channels
 *           (SSIMU2_PIPELINE_SPLIT only: the default pipeline never materialises these planes)
 * Only valid until that slot is reused (i.e. right after ssimu2_get_score). */
int ssimu2_debug_read(ssimu2_t *h, uint64_t ticket, int what, int scale, float *out, size_t out_floats);
/* Copy the per-strip partial sums of the pair `ticket` (same slot rule as ssimu2_debug_read) to host memory:
 * double[total_strips][3][6], channel x {ssim L1, ssim L4, artifact L1, artifact L4, detail L1, detail L4}, where an
 * L1 entry is the strip's sum of the map and an L4 entry the sum of its fourth power (k_finalize reduces them to the norms).
 * The strips of scale s are rows strip0[s] .. strip0[s] + n_strips[s] - 1 (ssimu2_debug_strips); out_doubles >= 18 * total. */
int ssimu2_debug_read_partials(ssimu2_t *h, uint64_t ticket, double *out, size_t out_doubles);
/* Strip geometry of the partial-sum table: per scale (nscales of ssimu2_get_info) the first row and the number of strips;
 * *strip_cols = columns per strip (strip k of a scale covers columns [k * cols, (k + 1) * cols) of that scale). */
int ssimu2_debug_strips(const ssimu2_t *h, uint32_t strip0[6], uint32_t n_strips[6], uint32_t *strip_cols);
/* Run the device arithmetic helpers over an array (host pointers) so the tests can compare them bit for
 * bit with libm / IEEE division:  op 0: out[i] = cbrtf(in[i]);  op 1: powf(in[i], y);  op 2: in[i] / y (f32);
 * op 3: `in` holds n (num, den) pairs of DOUBLES, `out` n doubles: num / den;
 * op 4: `in` holds n (num, den) pairs of floats: the V-pass quotient;
 * op 5 / 6: the unchecked hot-path forms of op 0 / 1 (positive normal arguments only). */
int ssimu2_debug_math(int op, const float *in, float y, float *out, size_t n);
/* Device time (ms) of the last completed batch per kernel: front-end, hpass (fused: k_hv), vpass, finalize. */
int ssimu2_last_batch_ms(ssimu2_t *h, float ms[4]);
/* Device time (ms, CUDA events on the batch's own stream) summed per kernel over every batch completed so far:
 * front-end, hpass (fused: k_hv), vpass, finalize; optional counters; reset != 0 clears them. */
int ssimu2_kernel_ms(ssimu2_t *h, double ms_total[4], uint64_t *batches, uint64_t *pairs, int reset);

#ifdef __cplusplus
}
#endif
#endif /* SSIMU2_B200_DEBUG_H */
