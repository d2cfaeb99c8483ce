// b4d_common.cuh — shared definitions for the sm_100a BM4D kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b4d.h"
#include "../../include/b4d_noise.h"

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
void b4d_launch_normalise_wm(const long long *numq, const uint32_t *gmap, const float *fallback, float *out, int D,
                             int H, int W, int nvol, int z0, int z1, float inv_qscale, const float kf[4],
                             cudaStream_t s);
void b4d_launch_quantize(const float *in, uint16_t *out, long long n, float offset_sub, float offset_add,
                         float step, cudaStream_t s);
void b4d_launch_quantize_trunc(const float *in, uint16_t *out, long long n, float offset_sub, float offset_add,
                               float step, cudaStream_t s);
void b4d_launch_normalise_q16(const long long *numq, const uint32_t *gmap, const float *fallback, uint16_t *q16, int D,
                              int H, int W, int nvol, int z0, int z1, float inv_qscale, const float kf[4],
                              float offset_sub, float offset_add, float step, int trunc, cudaStream_t s);
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
// coherence gate (b4d_coherence.cu): 23 sums per (patch, label slot), see there
void b4d_launch_coherence(const float *raw, const unsigned long long *labels, int D, int H, int W, long long npatch,
                          int lag, int radius, const double *w, double *x, double *sm, double *tmp,
                          unsigned long long *keys, int cap, double *sums, int *overflow, cudaStream_t s);
// analysis of a float32 volume for the matching map: partial[6*blocks] doubles
int b4d_analyze_blocks();
void b4d_launch_analyze(const float *in, long long n, double c, double *partial, cudaStream_t s);
// issue-rate microbenchmarks: returns lane-ops executed
double b4d_launch_pipe_bench(int which, int iters, unsigned *sink, cudaStream_t s);
