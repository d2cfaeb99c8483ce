/*
 * b4d_noise.h — noise-level estimation (DESIGN §3.11) and Poisson-Gaussian denoising through the generalized
 * Anscombe transform (§3.12) in libb4d.so, an extension of the C ABI of b4d.h.
 *
 * It has no counterpart in the CPU oracle library: the tests check the device result against a NumPy
 * restatement of the contract (tests/test_noise_sigma.py).  Conventions as in b4d.h.
 */
#ifndef B4D_NOISE_H_
#define B4D_NOISE_H_

#include "b4d.h"

#ifdef __cplusplus
extern "C" {
#endif

#define B4D_NOISE_HIST_BINS 262141 /* |d| <= 4 * 65535 */

/* Noise level of n equal-shape uint16 volumes (DESIGN §3.11): per tile of a C-order grid of `tile`
 * (even sides; NULL = one tile per volume), sigma / mad / cells, host arrays of n * tiles entries; `hist`
 * (NULL-able, host, 262141 x int64) receives the exact histogram of |d| over every cell of the call.
 * d is the unnormalised HHH Haar detail of each 2x2x2 cell at an even origin (cells of 8 zeros are skipped);
 * mad = median |d| (exact), sigma = mad / (sqrt(8) * 0.6744897501960817); a tile without cells gives NaN. */
int b4d_noise_sigma_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3],
                        const int64_t tile[3], double *sigma, double *mad, int64_t *cells,
                        int64_t *hist, int in_on_device);
/* The same statistics from a (summed) histogram; host arithmetic only. */
int b4d_noise_sigma_from_hist(const int64_t *hist, double *sigma, double *mad, int64_t *cells);

/* ---- Poisson-Gaussian noise (DESIGN §3.12) ---- */
#define B4D_NLF_MAX_BINS 64

/* Camera model z = gain * Poisson(lambda) + N(offset, read_sigma^2): gain > 0, read_sigma >= 0, all finite. */
typedef struct b4d_pg_model {
    double gain;
    double offset;
    double read_sigma;
} b4d_pg_model;

/* Noise-level function of n equal-shape uint16 volumes (one set of bins for the whole call).  Cells and d as in
 * b4d_noise_sigma_u16; s = sum of the cell's 8 voxels.  A cell is in bin k iff 8 e_k <= s < 8 e_{k+1} for the
 * nbins + 1 strictly increasing finite edges e (count units, 1 <= nbins <= 64).  Per bin (host arrays of nbins):
 * cells, level_sum = sum s, mad = median |d| (exact), sigma = mad / (sqrt(8) * 0.6744897501960817),
 * level = level_sum / (8 cells) (NaN without cells).  fit[2] = (a, b) of var = a * level + b by least squares
 * over the bins of at least min_cells (>= 1) cells, weighted by cells; NaN with fewer than 2 such bins, whose
 * number goes to *usable. */
int b4d_noise_level_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3], const double *edges,
                        int nbins, int64_t min_cells, int64_t *cells, int64_t *level_sum, double *mad,
                        double *sigma, double *level, double fit[2], int64_t *usable, int in_on_device);
/* Generalized Anscombe transform of n uint16 values -> float32 (forward), and the closed-form approximation of
 * its exact unbiased inverse, float32 -> float32.  Elementwise, any alignment. */
int b4d_gat_forward_u16(b4d_handle *h, const b4d_pg_model *model, const uint16_t *in, int64_t n, float *out,
                        int in_on_device, int out_on_device);
int b4d_gat_inverse_f32(b4d_handle *h, const b4d_pg_model *model, const float *in, int64_t n, float *out,
                        int in_on_device, int out_on_device);
/* Denoise n uint16 volumes under the model: inverse(denoise_f32(forward(z), sigma_vst)), sigma_vst > 0 (1 for an
 * exact model).  The q16 form writes the uint16 volume b4d_quantize_u16 (truncate = 0) or
 * b4d_quantize_trunc_u16 (truncate = 1) gives on that float32 result. */
int b4d_denoise_vst_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3],
                        const b4d_pg_model *model, float sigma_vst, float *out, int in_on_device, int out_on_device);
int b4d_denoise_vst_q16_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3],
                            const b4d_pg_model *model, float sigma_vst, float offset_sub, float offset_add,
                            float step, int truncate, uint16_t *out, int in_on_device, int out_on_device);

#ifdef __cplusplus
}
#endif
#endif /* B4D_NOISE_H_ */
