// b4d_common.cuh — shared definitions for the sm_100a BM4D kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

#include "../../include/b4d.h"
#include "../../include/b4d_noise.h"
#include "../../include/b4d_step_table.h"

// Kernels this host thread has enqueued.  A stage mark of the host pipeline books the kernels enqueued since the
// previous mark as that stage's launch count.  Per thread because the launchers do not see the handle; a call
// runs on one thread (the transfer threads only copy).
inline thread_local long long b4d_kernels_enqueued = 0;

// The one place that enqueues a kernel (every launcher goes through it, so every kernel is counted).
template <class... P, class... A>
inline void b4d_launch(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, A &&...args) {
    kernel<<<grid, block, smem, s>>>(std::forward<A>(args)...);
    ++b4d_kernels_enqueued;
}

#define B4D_L 4
#define B4D_LV 64
#define B4D_INVALID_KEY 0xFFFFFFFFu
#define B4D_FULL 0xFFFFFFFFu

// Geometry of one launch: `nvol` equal-shape volumes, reference-block origin
// lists per axis (device pointers).  All volumes share the lists.
struct B4dGeom {
    int D, H, W;
    int nvol;
    int nrz, nry, nrx;       // reference blocks per axis
    int tz, ty, tx;          // 4x4x4-reference tiles per axis
    const int *refz, *refy, *refx;
    long long vol_stride;    // voxels per volume
    long long refs_per_vol;
};

// Tables shared by the filter kernels; built on the host in float64 and rounded
// once, exactly as oracle/b4d_oracle.cpp make_tables() does.
struct B4dTables {
    float win[B4D_LV];   // (w[z]*w[y])*w[x], float32 products
    float kf[4];         // per-axis Kaiser factors w[n]: the normalise kernel convolves the weight map with them
    float tht[16];       // lambda*sigma*2^(m/2)
    // Wiener stage, unnormalised DCT butterflies: a raw coefficient with n odd positions (of x, y, z) at
    // group level l has the true value raw * S_n * 2^(-l/2), S_n = (1/2)^(3-n) c3^n, c3 = cos(3 pi/8)/sqrt 2.
    float wa[24];        // [n][l] = S_n 2^(-l/2): raw -> true (input of the attenuation)
    float wb[24];        // [n][l] = S_n^2 2^(-l): raw * W -> input of the unnormalised inverse butterflies
    float tq;            // 1 + sqrt 2 = c1 / c3
    float sigma2;
    // coloured noise (b4d_set_noise_model): relative variance nu_c = var_c / sigma^2 of every coefficient of the 3-D
    // transform of a 4^3 block of noise, in the kernels' coefficient order (z*4 + y)*4 + x-position
    float nu_ht[B4D_LV];   // Haar domain (stage 1)
    float nu_wie[B4D_LV];  // DCT domain (stage 2)
    float s2c[B4D_LV];     // sigma^2 nu_wie[c]
    float thc[B4D_LV * 6]; // [c][l] = lambda sigma sqrt(nu_ht[c]) 2^(m/2), m = 6 - n(c) + l
};

struct MatchParams {
    B4dGeom g;
    const uint16_t *u;   // matching image [nvol][D][H][W]
    const uint2 *s21;    // per block origin (K0): .x = energy sum(v^2) mod 2^32, .y = sum(v)
    uint32_t *cells;     // scratch: min | max << 16 per (plane, tile row, tile column): [nvol][D][ty][tx]
    uint32_t *tcls;      // scratch: class of every matcher tile (bit 16 byte tile + min in bits 0-15,
                         // bit 17 narrow), written by k_tile_class
    uint32_t tau;        // acceptance threshold (SSD <= tau)
    int K;               // max group size
    uint16_t *widx;      // [R][K] window index of each match
    uint8_t *cnt;        // [R] group size (power of two)
    uint32_t *ssd_out;   // optional [R][K] exact SSDs (instrumented matcher)
    long long tile0;     // first tile of this launch (set by the launcher)
    unsigned long long *stats;  // optional: [0] fallback refs, [1] wide tiles
    int use_tma;         // set by the launcher: the byte kernel stages its window with one TMA box load
    int use_tma_tab;      // general kernel: the {S2, S1} table arrives as one TMA box (W even)
};

struct FilterParams {
    B4dGeom g;
    const float *zf;     // noisy volume (float32)
    const float *basic;  // basic estimate (Wiener stage only)
    const uint16_t *widx;
    const uint8_t *cnt;
    int K;
    int Ns;
    int nseg;                    // z segments per column (set by the launcher)
    int seg0, nseg_launch;       // segments [seg0, seg0 + nseg_launch) belong to this launch
    float qscale;                // power of two: numerator terms are rint(wq * qscale * x), |.| < 2^39
    long long *numq;             // fixed-point numerator (order independent): sum of rint(wq * qscale * x)
    uint32_t *gmap;              // weight map: per block origin, the sum of the 20-bit group weights qg
    int psd;                     // coloured-noise tables are in effect (per-coefficient thresholds / attenuation)
#ifdef B4D_DEBUG_DUMP
    long long dbg_ref;           // developer builds: the Wiener-stage reference whose intermediates are printed
#endif
};

void b4d_launch_block_energy(const uint16_t *u, uint2 *s21, int D, int H, int W, int nvol, cudaStream_t s);
void b4d_launch_match(const MatchParams &p, int Ns, cudaStream_t s);
// the same in pieces (one volume arriving over PCIe plane by plane): block energies of origin planes
// [zo0, zo1); min/max of cell planes [cz0, cz1) and classification + matching of tiles [tile0, tile1)
void b4d_launch_block_energy_range(const uint16_t *u, uint2 *s21, int D, int H, int W, int nvol, int zo0, int zo1,
                                   cudaStream_t s);
void b4d_launch_match_range(const MatchParams &p, int Ns, int cz0, int cz1, long long tile0, long long tile1,
                            cudaStream_t s);
void b4d_launch_filter(const FilterParams &p, bool wiener, cudaStream_t s);
// the same in pieces: number of z segments (a multiple of `chunks` when the volume is deep enough,
// else the default), and the launch of segments [seg0, seg0 + count)
int b4d_filter_segments(const FilterParams &p, bool wiener, int chunks);
void b4d_launch_filter_segments(const FilterParams &p, bool wiener, int nseg, int seg0, int count, cudaStream_t s);
void b4d_upload_tables(const B4dTables &t, cudaStream_t s);

// misc kernels (b4d_misc.cu)
void b4d_launch_u16_to_f32(const uint16_t *in, float *out, long long n, unsigned *minmax, cudaStream_t s);
void b4d_launch_to_match(const float *in, uint16_t *out, long long n, float cf, float scale, int ishift,
                         cudaStream_t s);
void b4d_launch_u16_sub_offset(const uint16_t *in, const float *off, float *out, long long vol_stride, long long n,
                               unsigned *minmax, cudaStream_t s);
void b4d_launch_clip(float *x, long long n, float hi, cudaStream_t s);
void b4d_launch_add_scalar(float *x, long long n, float c, cudaStream_t s);
void b4d_launch_normalise_match(const long long *numq, const uint32_t *gmap, const float *fallback, float *out,
                                uint16_t *match, float mscale, int ishift, int D, int H, int W, int nvol,
                                float inv_qscale, const float kf[4], cudaStream_t s);
// weight-map contract: den = G (*) (kf x kf x kf) over planes [z0, z1) of every volume, out = num / den / qscale
// (with `epi`: the GAT inverse of that, see GatEpilogue)
struct GatEpilogue;
void b4d_launch_normalise_wm(const long long *numq, const uint32_t *gmap, const float *fallback, float *out, int D,
                             int H, int W, int nvol, int z0, int z1, float inv_qscale, const float kf[4],
                             const GatEpilogue *epi, cudaStream_t s);
void b4d_launch_quantize(const float *in, uint16_t *out, long long n, float offset_sub, float offset_add,
                         float step, cudaStream_t s);
void b4d_launch_quantize_trunc(const float *in, uint16_t *out, long long n, float offset_sub, float offset_add,
                               float step, cudaStream_t s);
void b4d_launch_normalise_q16(const long long *numq, const uint32_t *gmap, const float *fallback, uint16_t *q16, int D,
                              int H, int W, int nvol, int z0, int z1, float inv_qscale, const float kf[4],
                              float offset_sub, float offset_add, float step, int trunc, const GatEpilogue *epi,
                              cudaStream_t s);
// Per-tile quantizer steps (include/b4d_step_table.h, DESIGN §3 item 13) on the device: t[(iz * nty + iy) * ntx + ix]
// = {s, 65535 / s} (float32 division, as K7's __fdiv_rn) of tile (iz, iy, ix); plane z of a launch is global plane
// z0 + z.
struct StepTab {
    const float2 *t;
    int tz, ty, tx, nty, ntx;
    int z0;
};
// K6 + K7 fused with a step table (single volume)
void b4d_launch_normalise_qt16(const long long *numq, const uint32_t *gmap, const float *fallback, uint16_t *q16, int D,
                               int H, int W, int z0, int z1, float inv_qscale, const float kf[4], float offset_sub,
                               float offset_add, const StepTab &tab, int trunc, cudaStream_t s);
// standalone K7 with a step table, and its inverse, over the D x H x W planes of a launch
void b4d_launch_quantize_tiled(const float *in, uint16_t *out, int D, int H, int W, float offset_sub, float offset_add,
                               const StepTab &tab, int trunc, cudaStream_t s);
void b4d_launch_dequantize_tiled(const uint16_t *in, float *out, int D, int H, int W, float offset_sub,
                                 float offset_add, const StepTab &tab, cudaStream_t s);
void b4d_launch_hist(const uint16_t *in, long long n, unsigned long long *hist, cudaStream_t s);
// make_foreground_mask after the statistic: threshold + L1-ball dilation, per patch thr / off
void b4d_launch_fg_mask(const uint16_t *in, const float *off, const float *thr, int D, int H, int W, long long n,
                        int dilate, uint8_t *out, cudaStream_t s);
// K9: C-order chunk gather + 2-byte shuffle (+ per-chunk byte histograms [nchunks][2][256])
void b4d_launch_chunk_shuffle(const uint16_t *in, int D, int H, int W, int cz, int cy, int cx, uint8_t *out,
                              uint32_t *hist, cudaStream_t s);
// noise level (b4d_noise.cu): Haar-detail median per tile, DESIGN §3.11.  Cells are 2x2x2 at even origins, counted
// per axis (ncz, ncy, ncx); tiles are tcz x tcy x tcx cells, ntz x nty x ntx per volume, numbered over all volumes.
struct NoiseGeom {
    const uint16_t *in;
    long long vol_stride;  // voxels per volume
    int H, W;
    int ncz, ncy, ncx;
    int tcz, tcy, tcx;
    int ntz, nty, ntx;
    long long tile0;       // first tile of the launch (passes): scratch entries are relative to it
    int rows_per_cta, ctas_per_tile, warps;
};
// pass 1 (high digit) or 2 (low digit of the chosen bins) over `ntiles` tiles from g.tile0: hist[ntiles][1024]
void b4d_launch_noise_pass(const NoiseGeom &g, int pass, long long ntiles, uint32_t *hist, const uint32_t *sel,
                           cudaStream_t s);
// select 1 (sel[ntiles][5] = m, bin / rank of (m-1)/2, bin / rank of m/2) or 2 (res[ntiles][3] = a, b, m)
void b4d_launch_noise_select(int which, const uint32_t *hist, uint32_t *sel, uint32_t *res, long long ntiles,
                             cudaStream_t s);
// whole-call histogram of |d| over every cell of `nvol` volumes: hist[B4D_NOISE_HIST_BINS], accumulated
void b4d_launch_noise_hist(const NoiseGeom &g, long long nvol, unsigned long long *hist, cudaStream_t s);
// noise-level function (b4d_noise.cu, DESIGN §3.12): the same passes keyed by the intensity bin of each cell.
// thr[k] = ceil(8 e_k) clamped to [0, 524281] for k <= nb, INT32_MAX beyond: a cell of sum s is in bin k iff
// thr[k] <= s < thr[k + 1].  A launch covers bins [kb0, kb1).
constexpr int NLF_THR = 128;
struct NlfGeom {
    const uint16_t *in;
    long long vol_stride, nvol;
    int H, W;
    int ncz, ncy, ncx;
    int nb, kb0, kb1;
    int thr[NLF_THR];
};
// bins per launch of pass 1 / pass 2 (shared-memory histograms of 2 KB / 4 KB per bin)
int b4d_nlf_bins_per_launch(int pass);
// pass 1: hist[k][0, 512) and lsum[k] (sum s); pass 2: hist[k][0, 1024) from sel[k][5] of select 1
void b4d_launch_nlf_pass(const NlfGeom &g, int pass, uint32_t *hist, unsigned long long *lsum, const uint32_t *sel,
                         cudaStream_t s);
// generalized Anscombe transform (b4d_vst.cu, DESIGN §3.12): qq = (read_sigma / gain)^2, s15 = sqrt(1.5),
// c1 = 0.25 s15, c2 = 0.625 s15, all float64 from the host
struct GatParams {
    double gain, offset, qq, s15, c1, c2;
};
void b4d_launch_gat_forward(const uint16_t *in, float *out, long long n, const GatParams &p, cudaStream_t s);
// float32 result into `out`, or (q16 non-null) K7 of it into q16
void b4d_launch_gat_inverse(const float *in, float *out, uint16_t *q16, long long n, const GatParams &p,
                            float offset_sub, float offset_add, float step, int trunc, cudaStream_t s);
// The value set of a VST pass (DESIGN §3.12, map rule): list[i] = forward(vals[i]) for the m values, and the same
// value in table[vals[i]] (table: 65536 floats, NaN where no value was written).
void b4d_launch_gat_values(const uint16_t *vals, int m, const GatParams &p, float *list, float *table, cudaStream_t s);
// Forward with a known map: zf[i] = table[in[i]], match[i] = to_match(zf[i], cf, scale, ishift); *absent |= 1 when
// a value's entry is NaN (not in the value set).  `match` may be `in` (in place).
void b4d_launch_gat_forward_map(const uint16_t *in, const float *table, float *zf, uint16_t *match, long long n,
                                float cf, float scale, int ishift, unsigned *absent, cudaStream_t s);
// Epilogue of the last normalise of a VST pass: y = gat_inverse1(y + centre) (the add only when centre != 0).
struct GatEpilogue {
    GatParams p;
    float centre;
};

// K7: q = rint(clip((x - offset_sub + offset_add) / step, 0, 65535/step)).
// float32, clip BEFORE round, round-half-to-even: transforms.py:403-411.
__device__ __forceinline__ uint32_t quant1(float x, float osub, float oadd, float step, float hi, bool unit) {
    float v = __fadd_rn(__fsub_rn(x, osub), oadd);
    if (!unit) v = __fdiv_rn(v, step);
    v = fminf(fmaxf(v, 0.0f), hi);
    return (uint32_t)__float2int_rn(v);
}
// truncating variant: np.maximum(x, 0).astype(int) (evaluate.py:202) followed by the uint16 cast of
// compute_cratio (utils/img_util.py:420-423): toward zero, no upper clip, int64 -> uint16 wraps modulo 2^16
__device__ __forceinline__ uint32_t quant1_trunc(float x, float osub, float oadd, float step, float hi, bool unit) {
    (void)hi;
    float v = __fadd_rn(__fsub_rn(x, osub), oadd);
    if (!unit) v = __fdiv_rn(v, step);
    v = fmaxf(v, 0.0f);  // NaN -> 0
    return (uint32_t)(__float2ll_rz(v) & 0xFFFFll);
}
template <bool TRUNC>
__device__ __forceinline__ uint32_t quantq(float x, float osub, float oadd, float step, float hi, bool unit) {
    return TRUNC ? quant1_trunc(x, osub, oadd, step, hi, unit) : quant1(x, osub, oadd, step, hi, unit);
}
// GAT inverse of one value (DESIGN §3.12): float64, every operation in the order of the contract (-fmad=false)
__device__ __forceinline__ float gat_inverse1(float D, const GatParams &p) {
    const double d = (double)D;
    double lam = 0.0;
    if (!(d <= p.s15)) {  // P(sqrt(1.5)) = 0: the floor below is continuous; NaN takes this branch and gives 0
        const double r = 1.0 / d;
        const double P = 0.25 * d * d + p.c1 * r - 1.375 * r * r + p.c2 * r * r * r - 0.125;
        const double l = P - p.qq;
        lam = l > 0.0 ? l : 0.0;
    }
    return (float)(p.gain * lam + p.offset);
}
// Matching image: u = clamp(int(rint((v + cf) * scale)) + ishift, 0, 65535): the integer shift is applied after
// rounding so that rounding never depends on it.
__device__ __forceinline__ uint32_t to_match(float v, float cf, float scale, int ishift) {
    long long q = (long long)__float2ll_rn((v + cf) * scale) + ishift;
    q = min(max(q, 0ll), 65535ll);
    return (uint32_t)q;
}
// coherence gate (b4d_coherence.cu): 23 sums per (patch, label slot), see there
void b4d_launch_coherence(const float *raw, const unsigned long long *labels, int D, int H, int W, long long npatch,
                          int lag, int radius, const double *w, double *x, double *sm, double *tmp,
                          unsigned long long *keys, int cap, double *sums, int *overflow, cudaStream_t s);
// analysis of a float32 volume for the matching map: partial[6*blocks] doubles
int b4d_analyze_blocks();
void b4d_launch_analyze(const float *in, long long n, double c, double *partial, cudaStream_t s);
// issue-rate microbenchmarks: returns lane-ops executed
double b4d_launch_pipe_bench(int which, int iters, unsigned *sink, cudaStream_t s);
