/*
 * b4d_step_table.h — per-tile quantizer steps (DESIGN §3 item 13), an extension of the C ABI of b4d.h.
 *
 * A step table is a tile (tz, ty, tx), each side >= 1, a grid (ntz, nty, ntx) and steps[ntz][nty][ntx] (host,
 * float32).  The grid covers the whole volume (Z, H, W) in C order, anchored at (0, 0, 0) and ragged at the far faces
 * (the grid of K9's chunks and of b4d_noise_sigma_u16's tiles): nty = ceil(H / ty), ntx = ceil(W / tx).  The voxel at
 * GLOBAL (z, y, x) uses s = steps[z / tz][y / ty][x / tx].  Every step must be finite and >= 1; anything else is
 * B4D_ERR_INVALID before any device work.  The table is copied into a handle buffer on every call.
 *
 * Quantize: the uint16 result of a voxel is, bit for bit, what b4d_quantize_u16 (truncate = 0) or
 * b4d_quantize_trunc_u16 (truncate = 1) gives on it with step = s: a table whose entries all equal s reproduces the
 * scalar path.  Dequantize: x = ((float)q * s) + offset_sub - offset_add, each operation one float32 IEEE operation
 * in that order.
 *
 * b4d_quantize_tiled_u16 / b4d_dequantize_tiled_f32: planes [z_begin, z_begin + shape[0]) of a larger volume
 * (z_begin = 0 for a whole volume); ntz >= ceil((z_begin + shape[0]) / tz).
 * b4d_denoise_slab_qt16_u16: b4d_denoise_slab_q16_u16 with the table (a whole volume is the slab 0, D, 0, D), tile
 * rows indexed with global planes; ntz = ceil(z_total / tz).
 * b4d_slab_stage2_qt16: b4d_slab_stage2_q16 with the table, for the slab opened by b4d_slab_stage1_u16;
 * ntz = ceil(z_total / tz).  A VST slab is B4D_ERR_UNSUPPORTED.
 */
#ifndef B4D_STEP_TABLE_H_
#define B4D_STEP_TABLE_H_

#include "b4d.h"

#ifdef __cplusplus
extern "C" {
#endif

int b4d_quantize_tiled_u16(b4d_handle *h, const float *in, const int64_t shape[3], int64_t z_begin,
                           const int64_t tile[3], const int64_t grid[3], const float *steps, float offset_sub,
                           float offset_add, int truncate, uint16_t *out, int in_on_device, int out_on_device);
int b4d_dequantize_tiled_f32(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                             const int64_t tile[3], const int64_t grid[3], const float *steps, float offset_sub,
                             float offset_add, float *out, int in_on_device, int out_on_device);
int b4d_denoise_slab_qt16_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                              int64_t z_total, int64_t own_begin, int64_t own_end, float sigma, float offset_sub,
                              float offset_add, const int64_t tile[3], const int64_t grid[3], const float *steps,
                              int truncate, uint16_t *out, int in_on_device, int out_on_device);
int b4d_slab_stage2_qt16(b4d_handle *h, int64_t own_begin, int64_t own_end, float offset_sub, float offset_add,
                         const int64_t tile[3], const int64_t grid[3], const float *steps, int truncate,
                         uint16_t *out, int out_on_device);

#ifdef __cplusplus
}
#endif
#endif /* B4D_STEP_TABLE_H_ */
