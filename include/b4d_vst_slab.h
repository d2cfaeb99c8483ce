/*
 * b4d_vst_slab.h — z-slab forms of the Poisson-Gaussian (VST) path of b4d_noise.h (DESIGN §3.12, map rule), an
 * extension of the C ABI of b4d.h.
 *
 * A VST pass derives its matching map and centring from the set of uint16 values of the volume and its first voxel
 * alone.  A slab is given both for the WHOLE volume, so its owned planes equal those of b4d_denoise_vst_u16 on the
 * whole volume bit for bit (float32 and q16 output).  value_hist: host, 65536 x int64, counts of every uint16 value
 * of the whole volume (only > 0 matters: b4d_tile_stats' hist, or such histograms summed across ranks);
 * first_value: the whole volume's voxel (0, 0, 0).  B4D_ERR_INVALID for a NULL value_hist, a negative count,
 * value_hist[first_value] == 0, or a slab that holds a value whose count is 0.  Slab arguments and output as
 * b4d_denoise_slab_u16 / _q16_u16; b4d_slab_stage1_vst_u16 opens the slab of the two-call form, which
 * b4d_slab_basic_planes / _basic_ptr / _stage2_begin / _stage2 / _stage2_q16 complete (stage 2 ends in the inverse).
 */
#ifndef B4D_VST_SLAB_H_
#define B4D_VST_SLAB_H_

#include "b4d_noise.h"

#ifdef __cplusplus
extern "C" {
#endif

int b4d_denoise_slab_vst_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                             int64_t z_total, int64_t own_begin, int64_t own_end, const b4d_pg_model *model,
                             float sigma_vst, const int64_t *value_hist, int first_value, float *out, int in_on_device,
                             int out_on_device);
int b4d_denoise_slab_vst_q16_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                                 int64_t z_total, int64_t own_begin, int64_t own_end, const b4d_pg_model *model,
                                 float sigma_vst, const int64_t *value_hist, int first_value, float offset_sub,
                                 float offset_add, float step, int truncate, uint16_t *out, int in_on_device,
                                 int out_on_device);
int b4d_slab_stage1_vst_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                            int64_t z_total, const b4d_pg_model *model, float sigma_vst, const int64_t *value_hist,
                            int first_value, int in_on_device);

#ifdef __cplusplus
}
#endif
#endif /* B4D_VST_SLAB_H_ */
