/*
 * b4d_noise.h — noise-level estimation in libb4d.so (DESIGN §3.11), an extension of the C ABI of b4d.h.
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

#ifdef __cplusplus
}
#endif
#endif /* B4D_NOISE_H_ */
