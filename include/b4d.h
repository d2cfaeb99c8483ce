/*
 * b4d.h — C ABI of the B200-native BM4D denoise path (libb4d.so).
 *
 * What this boundary replaces in the reference (paths under /root/reference):
 *
 *   - `from bm4d import bm4d`           machine_learning/data_handling.py:12, evaluate.py:11
 *   - `teacher = bm4d(raw, sigma)`      machine_learning/data_handling.py:332, :926
 *   - `bm4d(noise, 10)`                 evaluate.py:202            (uint16 view in)
 *   - offset subtract before the call   machine_learning/data_handling.py:353-354
 *   - clip after the call               machine_learning/data_handling.py:333, :927
 *   - clip + rint + uint16              machine_learning/transforms.py:150-152, :409-411
 *   - low percentile of non-zero voxels machine_learning/transforms.py:433-438
 *   - median / MAD noise statistic      machine_learning/metrics.py:54-58
 *
 * The reference has no FFI of its own for this path: the arithmetic lives in
 * the closed third-party wheel bm4d==4.2.5 (uv.lock:387-400), bound by name at
 * import time.  The entry points below are what a ctypes binding for that call
 * needs; INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every function returns 0 on success or a negative b4d_status;
 *     b4d_last_error() returns a thread-local message for the last failure;
 *   - the caller owns every data buffer, the handle owns scratch and a stream;
 *   - pointers are host pointers unless the matching *_on_device flag is set;
 *   - volumes are C-order (z, y, x), x fastest, shape = {D, H, W};
 *   - one handle per (process, device); a handle is not thread-safe;
 *   - calls are synchronous: results are complete when the call returns.
 *
 * The same ABI is implemented by the CPU oracle (oracle/liboracle.so, test
 * infrastructure only) so one harness drives both.
 */
#ifndef B4D_H_
#define B4D_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B4D_ABI_VERSION 1

typedef enum b4d_status {
    B4D_OK = 0,
    B4D_ERR_INVALID = -1,     /* bad argument (shape, dtype contract, profile) */
    B4D_ERR_CUDA = -2,        /* a CUDA call failed; message names the call     */
    B4D_ERR_NOMEM = -3,       /* host or device allocation failed               */
    B4D_ERR_UNSUPPORTED = -4, /* valid request this build does not implement    */
    B4D_ERR_TOO_LARGE = -5    /* index space exceeds the ABI's integer width    */
} b4d_status;

/* Algorithm profile.  Defaults are SURVEY.md Appendix A; every constant the
 * closed bm4d binary may choose differently is a field here. */
typedef struct b4d_profile {
    int32_t abi;            /* B4D_ABI_VERSION                                         */
    int32_t block;          /* block side L; only 4 is implemented                     */
    int32_t step;           /* reference-block stride; only 3 is implemented           */
    int32_t search_ht;      /* search window side Ns (odd, 3..15), stage 1             */
    int32_t search_wie;     /* search window side Ns (odd, 3..15), stage 2             */
    int32_t k_ht;           /* max group size, stage 1 (power of two, <= 32)           */
    int32_t k_wie;          /* max group size, stage 2 (power of two, <= 32)           */
    int32_t stages;         /* 1 = hard-threshold stage only, 2 = + Wiener stage       */
    int32_t deterministic;  /* kept for ABI stability: aggregation is ALWAYS order-      *
                             * independent fixed point (bit-reproducible): dead field    */
    int32_t reserved0;
    float tau_ht;           /* match acceptance: SSD <= floor(tau*sigma^2*L^3)         */
    float tau_wie;
    float lambda_ht;        /* hard threshold: zero |c| < lambda*sigma                 */
    float kaiser_beta;      /* aggregation window; <= 0 selects an all-ones window     */
} b4d_profile;

/* Per-tile statistics (K8).  Semantics are exact: every field is what NumPy 2.x
 * returns on the same uint16 data cast to float32 (float32 virtual index and
 * interpolation included), widened to double. */
typedef struct b4d_stats {
    int64_t n;              /* voxels seen                                             */
    int64_t n_nonzero;      /* voxels > 0                                              */
    double offset;          /* percentile(x[x > 0], pct)       transforms.py:433-438   */
    double median;          /* median(x)                       metrics.py:55           */
    double mad;             /* median(|x - median|) + 1e-6     metrics.py:56           */
    double sigma;           /* 1.4826 * mad                    metrics.py:57           */
    double vmin;
    double vmax;
} b4d_stats;

typedef struct b4d_handle b4d_handle;

int b4d_version(void);
const char *b4d_last_error(void);
void b4d_default_profile(b4d_profile *p);

/* Create / destroy a handle bound to CUDA device `device` (ignored by the
 * oracle build).  `profile` may be NULL for the defaults. */
int b4d_create(int device, const b4d_profile *profile, b4d_handle **out);
void b4d_destroy(b4d_handle *h);
int b4d_set_profile(b4d_handle *h, const b4d_profile *profile);

/* Full BM4D denoise of `n` independent equal-shape volumes (n = 1 for one
 * patch).  Replaces bm4d.bm4d(z, sigma) at data_handling.py:332/:926 and
 * evaluate.py:202.  Output is float32, unclipped, same shape.
 *
 * u16: the filter runs on float(in); matching runs on the integers.
 * f32: the filter runs on `in`; matching runs on the integer image recovered
 *      from it (uint16 counts minus one scalar offset, data_handling.py:353-354)
 *      or, for non-integral data, on a 16-bit quantisation of it.            */
int b4d_denoise_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3],
                    float sigma, float *out, int in_on_device, int out_on_device);
int b4d_denoise_f32(b4d_handle *h, const float *in, int64_t n, const int64_t shape[3],
                    float sigma, float *out, int in_on_device, int out_on_device);

/* Voxels the handle processes per pass (default 1.25 Gi; scratch is about 45 bytes per voxel, so
 * the default needs ~60 GB of the 180 GB).  Batches are cut into passes of whole patches; ONE uint16
 * volume larger than a pass is denoised as consecutive z-slabs with halos on the same GPU
 * (b4d_denoise_u16 does this itself; the result equals the one-pass result bit for bit).
 * 0 restores the default. */
int b4d_set_pass_voxels(b4d_handle *h, int64_t voxels);

/* Volume size (voxels) from which the host transfers of one volume or slab are pipelined against
 * the kernels (chunked upload behind the stage-1 matcher, chunked stage 2 with copy-out of the
 * finished planes).  Default 2^26: below it the chunked launches under-fill the GPU and the
 * transfers are negligible.  The result never depends on it. */
int b4d_set_pipeline_min_voxels(b4d_handle *h, int64_t voxels);

/* Training targets for `n` equal-shape uint16 patches in one call — the core of
 * `_sample_counts` (data_handling.py:315-354) batched:
 *     raw     = float32(in) - offsets[i]                 data_handling.py:353-354
 *     teacher = clip(bm4d(raw, sigma), 0, max_count)     data_handling.py:332-333
 * `offsets` is a HOST array of n per-patch background offsets.  `raw_out` may be NULL.
 * Equal, bit for bit, to b4d_denoise_f32 on each raw patch followed by the clip: the counts
 * go over PCIe as uint16 (2 B/voxel), the subtraction and the clip run on the device. */
int b4d_targets_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3],
                    const float *offsets, float sigma, float max_count, float *raw_out,
                    float *teacher_out, int in_on_device, int out_on_device);

/* One z-slab of a larger volume (SURVEY §8e).  `in` holds global planes
 * [z_begin, z_begin + shape[0]) of a volume with `z_total` planes; reference
 * blocks sit on the GLOBAL grid and only those whose search window lies inside
 * the slab are processed.  `out` receives planes [own_begin, own_end) (global
 * numbering), own_end - own_begin planes of H*W floats.  Exact (equal to the
 * whole-volume result) when the slab extends 2*(Ns-1+L-1) planes beyond the
 * owned range on each interior face. */
int b4d_denoise_slab_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3],
                         int64_t z_begin, int64_t z_total, int64_t own_begin, int64_t own_end,
                         float sigma, float *out, int in_on_device, int out_on_device);

/* The same slab in two calls with ONE neighbour exchange in between (SURVEY §8e, "one
 * exchange step"): the slab then needs only (Ns-1+L-1) = 13 halo planes per interior face
 * instead of 26.
 *   1. b4d_slab_stage1_u16   stage 1 on the slab; the basic estimate stays on the device.
 *      It is exact on the planes at least 13 inside the slab's interior faces.
 *   2. b4d_slab_basic_planes copies planes of the basic estimate out of (to_handle = 0) or
 *      into (to_handle = 1) the handle, slab-local plane numbering: every rank sends its
 *      exact planes next to a face and overwrites its halo planes with the neighbour's.
 *   3. b4d_slab_stage2       stage 2 on the completed basic estimate; `out` receives the
 *      owned planes [own_begin, own_end) (global numbering).
 * Equal, bit for bit, to the whole-volume result. */
int b4d_slab_stage1_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                        int64_t z_total, float sigma, int in_on_device);
int b4d_slab_basic_planes(b4d_handle *h, int64_t plane0, int64_t nplanes, float *buf, int to_handle,
                          int buf_on_device);
int b4d_slab_stage2(b4d_handle *h, int64_t own_begin, int64_t own_end, float *out, int out_on_device);
/* Optional, between 1 and 3, for callers that exchange planes device to device:
 *   b4d_slab_basic_ptr      device pointer to the basic estimate of the open slab, [D][H][W] float32 — a neighbour
 *                           exchange (NCCL point-to-point) may read the owned planes and write the halo planes in place;
 *   b4d_slab_stage2_begin   launches, without waiting, the part of the stage-2 front end (matching image, block
 *                           energies, tile classification, matching) that reads owned planes only, so that the
 *                           exchange overlaps it; b4d_slab_stage2 then does the rest.  The result is unchanged. */
float *b4d_slab_basic_ptr(b4d_handle *h);
int b4d_slab_stage2_begin(b4d_handle *h, int64_t own_begin, int64_t own_end);
/* the same with the fused quantizer (see b4d_denoise_q16_u16) */
int b4d_slab_stage2_q16(b4d_handle *h, int64_t own_begin, int64_t own_end, float offset_sub,
                        float offset_add, float step, int truncate, uint16_t *out, int out_on_device);

/* Instrumented stage-1 matcher (bit-exactness test, BASELINE config 3).
 * R = number of reference blocks, K = profile.k_ht.  Host pointers.
 *   idx[R*K]   linear candidate origin (z*H' + y)*W' + x, H' = H-L+1, W' = W-L+1; -1 = unused
 *   ssd[R*K]   exact integer SSD; UINT64_MAX = unused
 *   count[R]   group size actually used (power of two)                        */
int b4d_match_stage1(b4d_handle *h, const uint16_t *in, const int64_t shape[3], float sigma,
                     int32_t *idx, uint64_t *ssd, int32_t *count);
int64_t b4d_num_refs(const int64_t shape[3]);

/* Fused offset-subtract + clip + (noise-scaled) quantize, K7:
 *   q = rint(clip((x - offset_sub + offset_add) / step, 0, 65535 / step)) -> uint16
 * At step = 1, offset_sub = 0 this is transforms.py:403-411 bit for bit. */
int b4d_quantize_u16(b4d_handle *h, const float *in, int64_t n, float offset_sub,
                     float offset_add, float step, uint16_t *out, int in_on_device,
                     int out_on_device);
/* The truncating variant the evaluator uses: np.maximum(x, 0).astype(int) (evaluate.py:202) followed by the
 * uint16 cast of compute_cratio (utils/img_util.py:420-423):
 *   q = uint16(int64(trunc(max((x - offset_sub + offset_add) / step, 0))))   toward zero, no upper clip,
 *   wrapping modulo 2^16 as the NumPy cast does; NaN gives 0. */
int b4d_quantize_trunc_u16(b4d_handle *h, const float *in, int64_t n, float offset_sub,
                           float offset_add, float step, uint16_t *out, int in_on_device,
                           int out_on_device);

/* Denoise -> offset -> quantize in one call (K6 + K7 fused: the float32 result is never stored, 2 bytes per
 * voxel leave the device instead of 4).  Equal, bit for bit, to b4d_quantize_u16 / b4d_quantize_trunc_u16
 * (truncate != 0) applied to the output of the matching denoise call.  Needs profile.stages = 2. */
int b4d_denoise_slab_q16_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                             int64_t z_total, int64_t own_begin, int64_t own_end, float sigma,
                             float offset_sub, float offset_add, float step, int truncate, uint16_t *out,
                             int in_on_device, int out_on_device);
int b4d_denoise_q16_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], float sigma,
                        float offset_sub, float offset_add, float step, int truncate, uint16_t *out,
                        int in_on_device, int out_on_device);

/* Intensity foreground mask of `n` equal-shape uint16 patches — make_foreground_mask
 * (machine_learning/metrics.py:32-61), the mask both datasets fall back to when a patch has no
 * annotation (data_handling.py:444, :928-929), on raw = float32(in) - offsets[i]
 * (data_handling.py:353-354):
 *     med = median(raw); mad = median(|raw - med|) + 1e-6; sigma = 1.4826 * mad      (float32)
 *     mask = raw > med + k * sigma, then `dilate` iterations of 6-neighbour binary dilation
 * `offsets` is a HOST array of n floats; `out` receives n * voxels bytes of 0 / 1.
 * The medians are exact (65 536-bin histogram per patch); the result equals the reference's
 * function bit for bit under NumPy 2 scalar rules (tests/golden/reference_masks.npz). */
int b4d_foreground_mask_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3],
                            const float *offsets, float k, int dilate, uint8_t *out,
                            int in_on_device, int out_on_device);

/* K9 — chunking + byte shuffle ahead of the chunk codec (SURVEY 8f row 2, first step).
 * The volume is cut the way compute_cratio does (utils/img_util.py:427-438): a C-order grid of
 * `chunk`-shaped pieces, ragged at the far faces, each piece made contiguous.  Each piece is then
 * byte-shuffled as Blosc SHUFFLE does for 2-byte items (evaluate.py:40): all low bytes, then all
 * high bytes.  `out` (2 * voxels bytes, NULL-able) receives the pieces back to back in grid order;
 * piece (iz,iy,ix) starts at byte 2 * (z0*H*W + dz*(y0*W + dy*x0)).  `hist` (NULL-able) receives
 * [pieces][2][256] uint32 counts of the byte values of the low and the high plane — the input of
 * an order-0 entropy estimate of the compressed size.  `out_on_device` applies to both outputs. */
int b4d_chunk_shuffle_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3],
                          const int64_t chunk[3], uint8_t *out, uint32_t *hist, int in_on_device,
                          int out_on_device);

/* Per-tile statistics, K8.  Also returns the exact 65536-bin histogram when
 * `hist` is non-NULL (host pointer, 65536 x int64) — that histogram is the
 * payload ranks allgather to agree on a global offset / sigma. */
int b4d_tile_stats(b4d_handle *h, const uint16_t *in, int64_t n, double pct, b4d_stats *out,
                   int64_t *hist, int in_on_device);
/* The same statistics from an exact 65 536-bin histogram of counts (e.g. the sum of the per-slab histograms the
 * ranks all-gather): host arithmetic only, no device work. */
int b4d_stats_from_hist(const int64_t *hist, double pct, b4d_stats *out);

/* The last public denoise call as a whole (every chunk, pass and slab of it; the two-call slab form from
 * b4d_slab_stage1_u16 to b4d_slab_stage2), per kernel family (B4D_T_* below): ms = device time in milliseconds
 * (CUDA events on the handle's stream), launches = the kernels enqueued in the intervals that family books.
 * Memsets and copies are not launches.  A few kernels are booked to no family: the add-back of the DC shift of
 * centred float input, the clip and offset subtraction of b4d_targets_u16, the block energies of
 * b4d_match_stage1. */
#define B4D_T_PREP 0
#define B4D_T_MATCH1 1
#define B4D_T_FILTER1 2
#define B4D_T_NORM1 3
#define B4D_T_MATCH2 4
#define B4D_T_FILTER2 5
#define B4D_T_NORM2 6
#define B4D_T_K0 7 /* block energies (K0) where they run as a launch of their own; inside PREP otherwise */
#define B4D_T_COUNT 8
int b4d_last_timings(b4d_handle *h, float ms[B4D_T_COUNT], int64_t launches[B4D_T_COUNT]);

/* The CUDA stream (cudaStream_t, as void *) every kernel and copy of this handle is
 * enqueued on — for callers that time with CUDA events or order their own work after
 * a call.  NULL for the CPU oracle build. */
void *b4d_stream(b4d_handle *h);

/* Diagnostics of the matching launches of the last public call, summed over all of them (as b4d_last_timings):
 * out[0] = reference blocks that
 * took the survivor-list overflow fallback, out[1] = tiles on the uint64 path,
 * out[2] = reference blocks on the exact-but-slow selection, out[3] = tiles matched
 * on the byte (dp4a) path. */
int b4d_last_match_stats(b4d_handle *h, uint64_t out[4]);

/* Measured issue-rate peaks on this device (shipped microbenchmark):
 *   out[0] = IMAD lane-ops/s, out[1] = IADD3 lane-ops/s,
 *   out[2] = dependent (sub, mad) pair stream in lane-ops/s (2 per pair),
 *   out[3] = FFMA lane-ops/s.                                                */
int b4d_measure_pipe_peaks(b4d_handle *h, double out[4]);

/* Coloured (spatially correlated) noise — the array form of bm4d's `sigma_psd` argument.  The caller reduces the
 * noise PSD to the relative variance nu_c = var_c / sigma^2 of each of the 64 coefficients of the 3-D block
 * transform of pure noise, for the stage-1 transform (Haar = bior1.5 at length 4) and the stage-2 transform
 * (DCT-II), coefficient order (z*4 + y)*4 + x with the positions of oracle/b4d_oracle.cpp; `sigma` of the following
 * denoise calls is the root of the mean noise variance.  Then: hard threshold lambda sigma sqrt(nu_c), weight
 * 1 / sum of nu_c over the retained coefficients; Wiener W = y^2 / (y^2 + sigma^2 nu_c), weight 1 / sum W^2 nu_c;
 * matching threshold tau sigma^2 64.  nu = 1 everywhere is the white model (bit-identical to NULL, NULL, which
 * switches the model off).  Search windows above 11 are not supported with a coloured model. */
int b4d_set_noise_model(b4d_handle *h, const float nu_ht[64], const float nu_wie[64]);

/* The spatial-coherence gate that precedes BM4D in the sampler (machine_learning/metrics.py:189-260
 * patch_has_incoherent_segment, with local_autocorr :64-112 and highfreq_energy_fraction :115-155; call site
 * data_handling.py:398-407), for `n` equal-shape patches: raw float32 counts, labels uint64 (0 = background).
 *   reject[i] = 1 when some segment of patch i with at least min_segment_voxels voxels has a lag-`lag`
 *   autocorrelation below min_autocorr AND a high-frequency energy fraction above max_highfreq_frac.
 * Optional per-segment scores (NULL to skip): seg[i * max_segments + j], j < seg_count[i], in no particular order. */
typedef struct b4d_segment_score {
    uint64_t label;
    int64_t voxels;
    double autocorr;   /* 1.0 when it cannot be measured, as the reference returns */
    double highfreq;   /* 0.0 when the segment's variance is degenerate            */
} b4d_segment_score;
int b4d_coherence_gate(b4d_handle *h, const float *raw, const uint64_t *labels, int64_t n, const int64_t shape[3],
                       double min_autocorr, double max_highfreq_frac, int64_t min_segment_voxels,
                       double smooth_sigma, int lag, uint8_t *reject, b4d_segment_score *seg,
                       int64_t max_segments, int64_t *seg_count, int in_on_device);

/* Diagnostics: the fixed-point aggregation state the LAST filter stage of the last single-volume call left
 * behind, copied to host arrays of n = D*H*W entries: numq = sum of the rounded numerator terms per voxel,
 * wmap = sum of the 20-bit group weights per block origin.  The tests compare both with the oracle mirror's,
 * integer for integer, which localises a difference to a reference block.  No reference-side counterpart. */
int b4d_debug_accumulators(b4d_handle *h, int64_t *numq, int64_t *wmap, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* B4D_H_ */
