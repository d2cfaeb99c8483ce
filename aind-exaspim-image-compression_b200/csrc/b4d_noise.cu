// b4d_noise.cu — noise level from the finest 3-D Haar detail (DESIGN §3.11).
//
// A cell is a 2x2x2 block at an even origin; its detail d = sum (-1)^(i+j+k) v[z+i, y+j, x+k] is the unnormalised
// HHH Haar coefficient, an integer with |d| <= 262140.  Per tile the median of |d| is found exactly by a two-pass
// radix select: pass 1 histograms the high digit |d| >> 9 (512 bins), a warp per tile finds the bins of the two
// middle ranks, pass 2 histograms the low 9 bits of the cells in those bins, a warp per tile reads the ranks off.
// Each pass reads the input once (2 B per voxel).
//
// Traversal: a CTA takes a run of cell rows (fixed z, y) of one tile, a warp one row at a time, lane = cell along
// x, so consecutive lanes read consecutive 4-byte words (W even, 4-byte aligned base) or 2-byte pairs otherwise.
#include "b4d_common.cuh"

namespace {

constexpr int NZ_FULL_HOT = 8192;  // shared partial of the whole-call histogram: |d| below this (noise lives there)

// |d| of the cell at (cz, cy, cx) of volume `vol`; `zero` = all 8 voxels are 0 (padding, not data)
template <bool WIDE>
__device__ __forceinline__ uint32_t cell_abs_detail(const uint16_t *__restrict__ vol, int H, int W, int cz, int cy,
                                                    int cx, bool &zero) {
    const long long plane = (long long)H * W;
    const uint16_t *p = vol + (2ll * cz * H + 2ll * cy) * W + 2ll * cx;
    int a0, b0, a1, b1, a2, b2, a3, b3;
    if (WIDE) {
        const uint32_t w0 = __ldcs(reinterpret_cast<const unsigned int *>(p));
        const uint32_t w1 = __ldcs(reinterpret_cast<const unsigned int *>(p + W));
        const uint32_t w2 = __ldcs(reinterpret_cast<const unsigned int *>(p + plane));
        const uint32_t w3 = __ldcs(reinterpret_cast<const unsigned int *>(p + plane + W));
        zero = (w0 | w1 | w2 | w3) == 0u;
        a0 = (int)(w0 & 0xFFFFu), b0 = (int)(w0 >> 16);
        a1 = (int)(w1 & 0xFFFFu), b1 = (int)(w1 >> 16);
        a2 = (int)(w2 & 0xFFFFu), b2 = (int)(w2 >> 16);
        a3 = (int)(w3 & 0xFFFFu), b3 = (int)(w3 >> 16);
    } else {
        a0 = __ldcs(p), b0 = __ldcs(p + 1);
        a1 = __ldcs(p + W), b1 = __ldcs(p + W + 1);
        a2 = __ldcs(p + plane), b2 = __ldcs(p + plane + 1);
        a3 = __ldcs(p + plane + W), b3 = __ldcs(p + plane + W + 1);
        zero = (a0 | b0 | a1 | b1 | a2 | b2 | a3 | b3) == 0;
    }
    // sign of row (i, j) is (-1)^(i+j), of the x pair (+, -)
    const int d = (a0 - b0) - (a1 - b1) - (a2 - b2) + (a3 - b3);
    return (uint32_t)(d < 0 ? -d : d);
}

// One histogram increment per lane with `ok`; lanes that add to the same bin are merged first, so that a warp
// whose cells share a bin (flat background, bin 0 of the high digit) costs one shared atomic instead of 32.
__device__ __forceinline__ void warp_hist_add(uint32_t *sh, uint32_t bin, bool ok) {
    const uint32_t peers = __match_any_sync(B4D_FULL, ok ? bin : 0xFFFFFFFFu);
    if (ok && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&sh[bin], (uint32_t)__popc(peers));
}

// Cell range of one tile: cells [c0, c1) per axis of volume `vol`.
struct TileCells {
    const uint16_t *vol;
    int cz0, cy0, cx0, nrz, nry, nrx;
};
__device__ __forceinline__ TileCells tile_cells(const NoiseGeom &g, long long t) {
    const long long per_vol = (long long)g.ntz * g.nty * g.ntx;
    const long long v = t / per_vol;
    const long long lt = t - v * per_vol;
    const int ix = (int)(lt % g.ntx), iy = (int)((lt / g.ntx) % g.nty), iz = (int)(lt / ((long long)g.ntx * g.nty));
    TileCells c;
    c.vol = g.in + v * g.vol_stride;
    c.cz0 = iz * g.tcz, c.cy0 = iy * g.tcy, c.cx0 = ix * g.tcx;
    c.nrz = max(0, min(g.tcz, g.ncz - c.cz0));
    c.nry = max(0, min(g.tcy, g.ncy - c.cy0));
    c.nrx = max(0, min(g.tcx, g.ncx - c.cx0));
    return c;
}

// Passes 1 and 2.  PASS 1: bins = |d| >> 9 into hist[t][0, 512).  PASS 2: the low 9 bits of the cells whose high
// digit is the bin of rank a (hist[t][0, 512)) or, when different, of rank b (hist[t][512, 1024)).
template <int PASS, bool WIDE>
__global__ void __launch_bounds__(256) k_noise_pass(NoiseGeom g, uint32_t *__restrict__ hist,
                                                    const uint32_t *__restrict__ sel) {
    constexpr int NB = PASS == 1 ? 512 : 1024;
    __shared__ uint32_t sh[NB];
    const long long tl = blockIdx.x / g.ctas_per_tile;  // tile of this CTA, relative to the launch
    const int part = (int)(blockIdx.x - tl * g.ctas_per_tile);
    const TileCells c = tile_cells(g, g.tile0 + tl);
    const int rows = c.nrz * c.nry;
    const int r0 = part * g.rows_per_cta, r1 = min(rows, r0 + g.rows_per_cta);
    if (r0 >= r1) return;  // uniform over the CTA
    uint32_t bin_a = 0, bin_b = 0;
    if (PASS == 2) {
        const uint32_t *s = sel + tl * 5;
        if (s[0] == 0u) return;  // no cell in this tile
        bin_a = s[1];
        bin_b = s[3];
    }
    for (int i = threadIdx.x; i < NB; i += blockDim.x) sh[i] = 0u;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int r = r0 + warp; r < r1; r += nwarps) {
        const int cz = c.cz0 + r / c.nry, cy = c.cy0 + r % c.nry;
        for (int x = 0; x < c.nrx; x += 64) {  // two cells per lane in flight
            const bool in0 = x + lane < c.nrx, in1 = x + 32 + lane < c.nrx;
            bool z0 = true, z1 = true;
            uint32_t d0 = 0, d1 = 0;
            if (in0) d0 = cell_abs_detail<WIDE>(c.vol, g.H, g.W, cz, cy, c.cx0 + x + lane, z0);
            if (in1) d1 = cell_abs_detail<WIDE>(c.vol, g.H, g.W, cz, cy, c.cx0 + x + 32 + lane, z1);
            if (PASS == 1) {
                warp_hist_add(sh, d0 >> 9, in0 && !z0);
                warp_hist_add(sh, d1 >> 9, in1 && !z1);
            } else {
                const uint32_t h0 = d0 >> 9, h1 = d1 >> 9;
                warp_hist_add(sh, (h0 == bin_a ? 0u : 512u) + (d0 & 511u),
                              in0 && !z0 && (h0 == bin_a || h0 == bin_b));
                warp_hist_add(sh, (h1 == bin_a ? 0u : 512u) + (d1 & 511u),
                              in1 && !z1 && (h1 == bin_a || h1 == bin_b));
            }
        }
    }
    __syncthreads();
    uint32_t *gh = hist + tl * 1024;
    for (int i = threadIdx.x; i < NB; i += blockDim.x)
        if (sh[i]) atomicAdd(&gh[i], sh[i]);
}

// Bin of 0-based rank k in the 512 bins h (k < total), and the rank left inside that bin.  Lane l holds bins
// [16 l, 16 l + 16); `excl` is the count below them.
__device__ __forceinline__ void warp_find_rank(const uint32_t (&v)[16], uint32_t excl, uint32_t incl, uint32_t k,
                                               uint32_t &bin, uint32_t &rem) {
    const int lane = threadIdx.x & 31;
    const uint32_t own = __ballot_sync(B4D_FULL, excl <= k && k < incl);
    const int src = __ffs(own) - 1;
    uint32_t b = 0, r = 0;
    if (lane == src) {
        uint32_t c = excl;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            if (k >= c && k < c + v[i]) {
                b = 16u * lane + i;
                r = k - c;
            }
            c += v[i];
        }
    }
    bin = __shfl_sync(B4D_FULL, b, src);
    rem = __shfl_sync(B4D_FULL, r, src);
}

__device__ __forceinline__ void warp_load_scan(const uint32_t *h, uint32_t (&v)[16], uint32_t &excl,
                                               uint32_t &incl, uint32_t &total) {
    const int lane = threadIdx.x & 31;
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        v[i] = h[16 * lane + i];
        s += v[i];
    }
    incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(B4D_FULL, incl, o);
        if (lane >= o) incl += t;
    }
    excl = incl - s;
    total = __shfl_sync(B4D_FULL, incl, 31);
}

// Select 1: one warp per tile.  sel[t] = {m, bin_a, rem_a, bin_b, rem_b} for the ranks a = (m-1)/2, b = m/2.
__global__ void __launch_bounds__(256) k_noise_select1(const uint32_t *__restrict__ hist, uint32_t *__restrict__ sel,
                                                       long long ntiles) {
    const long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t >= ntiles) return;  // uniform over the warp
    uint32_t v[16], excl, incl, m;
    warp_load_scan(hist + t * 1024, v, excl, incl, m);
    uint32_t ba = 0, ra = 0, bb = 0, rb = 0;
    if (m) {
        warp_find_rank(v, excl, incl, (m - 1u) / 2u, ba, ra);
        warp_find_rank(v, excl, incl, m / 2u, bb, rb);
    }
    if ((threadIdx.x & 31) == 0) {
        uint32_t *s = sel + t * 5;
        s[0] = m, s[1] = ba, s[2] = ra, s[3] = bb, s[4] = rb;
    }
}

// Select 2: one warp per tile.  res[t] = {a, b, m}: the two middle order statistics of |d| and the cell count.
__global__ void __launch_bounds__(256) k_noise_select2(const uint32_t *__restrict__ hist,
                                                       const uint32_t *__restrict__ sel, uint32_t *__restrict__ res,
                                                       long long ntiles) {
    const long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t >= ntiles) return;
    const uint32_t *s = sel + t * 5;
    const uint32_t m = s[0];
    uint32_t a = 0, b = 0;
    if (m) {
        uint32_t v[16], excl, incl, tot, low, rem;
        warp_load_scan(hist + t * 1024, v, excl, incl, tot);
        warp_find_rank(v, excl, incl, s[2], low, rem);
        a = (s[1] << 9) | low;
        if (s[3] != s[1]) warp_load_scan(hist + t * 1024 + 512, v, excl, incl, tot);
        warp_find_rank(v, excl, incl, s[4], low, rem);
        b = (s[3] << 9) | low;
    }
    if ((threadIdx.x & 31) == 0) {
        uint32_t *o = res + t * 3;
        o[0] = a, o[1] = b, o[2] = m;
    }
}

// Whole-call histogram of |d| (262 141 bins): a warp per cell row over every row of every volume; bins below
// NZ_FULL_HOT in a shared partial flushed once per CTA, the tail straight to global 64-bit atomics.
template <bool WIDE>
__global__ void __launch_bounds__(256) k_noise_hist(NoiseGeom g, long long nvol, unsigned long long *__restrict__ hist) {
    __shared__ uint32_t sh[NZ_FULL_HOT];
    for (int i = threadIdx.x; i < NZ_FULL_HOT; i += blockDim.x) sh[i] = 0u;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long rows_per_vol = (long long)g.ncz * g.ncy, rows = rows_per_vol * nvol;
    const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += nw) {
        const long long v = r / rows_per_vol;
        const int rr = (int)(r - v * rows_per_vol);
        const int cz = rr / g.ncy, cy = rr % g.ncy;
        const uint16_t *vol = g.in + v * g.vol_stride;
        for (int x = 0; x < g.ncx; x += 64) {
            const bool in0 = x + lane < g.ncx, in1 = x + 32 + lane < g.ncx;
            bool z0 = true, z1 = true;
            uint32_t d0 = 0, d1 = 0;
            if (in0) d0 = cell_abs_detail<WIDE>(vol, g.H, g.W, cz, cy, x + lane, z0);
            if (in1) d1 = cell_abs_detail<WIDE>(vol, g.H, g.W, cz, cy, x + 32 + lane, z1);
            const bool ok0 = in0 && !z0, ok1 = in1 && !z1;
            warp_hist_add(sh, d0, ok0 && d0 < NZ_FULL_HOT);
            warp_hist_add(sh, d1, ok1 && d1 < NZ_FULL_HOT);
            if (ok0 && d0 >= NZ_FULL_HOT) atomicAdd(&hist[d0], 1ull);
            if (ok1 && d1 >= NZ_FULL_HOT) atomicAdd(&hist[d1], 1ull);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NZ_FULL_HOT; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], (unsigned long long)sh[i]);
}

int sm_count() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

bool wide_ok(const NoiseGeom &g) { return (g.W & 1) == 0 && (reinterpret_cast<uintptr_t>(g.in) & 3) == 0; }

}  // namespace

void b4d_launch_noise_pass(const NoiseGeom &g, int pass, long long ntiles, uint32_t *hist, const uint32_t *sel,
                           cudaStream_t s) {
    const unsigned blocks = (unsigned)(ntiles * g.ctas_per_tile);
    const int threads = 32 * g.warps;
    const bool w = wide_ok(g);
    if (pass == 1) {
        if (w) k_noise_pass<1, true><<<blocks, threads, 0, s>>>(g, hist, sel);
        else k_noise_pass<1, false><<<blocks, threads, 0, s>>>(g, hist, sel);
    } else {
        if (w) k_noise_pass<2, true><<<blocks, threads, 0, s>>>(g, hist, sel);
        else k_noise_pass<2, false><<<blocks, threads, 0, s>>>(g, hist, sel);
    }
}

void b4d_launch_noise_select(int which, const uint32_t *hist, uint32_t *sel, uint32_t *res, long long ntiles,
                             cudaStream_t s) {
    const unsigned blocks = (unsigned)((ntiles + 7) / 8);
    if (which == 1) k_noise_select1<<<blocks, 256, 0, s>>>(hist, sel, ntiles);
    else k_noise_select2<<<blocks, 256, 0, s>>>(hist, sel, res, ntiles);
}

void b4d_launch_noise_hist(const NoiseGeom &g, long long nvol, unsigned long long *hist, cudaStream_t s) {
    const long long rows = (long long)g.ncz * g.ncy * nvol;
    long long blocks = (rows + 7) / 8;
    if (blocks > 4ll * sm_count()) blocks = 4ll * sm_count();
    if (wide_ok(g)) k_noise_hist<true><<<(unsigned)blocks, 256, 0, s>>>(g, nvol, hist);
    else k_noise_hist<false><<<(unsigned)blocks, 256, 0, s>>>(g, nvol, hist);
}
