// b4d_coherence.cu — the spatial-coherence gate that runs immediately before BM4D in the sampler
// (machine_learning/metrics.py:64-260: local_autocorr, highfreq_energy_fraction,
// patch_has_incoherent_segment; called at data_handling.py:398-407), on the device, for a batch of patches.
//
// Per segment (label id) of a patch the reference needs
//   * the lag-`lag` Pearson correlation along each axis over voxel pairs that both carry the label, and
//   * var(raw - gaussian_filter(raw)) / var(raw) over the segment's voxels,
// all in float64.  Both follow from 23 sums per segment (n, sum v, sum v^2, sum h, sum h^2 and per axis n,
// sum x, sum y, sum x^2, sum y^2, sum xy), which the kernels accumulate; the host turns them into the two scores
// and the reject decision with the reference's own formulas and edge rules.  The voxel values are centred on the
// patch's first voxel before anything is summed (every statistic is shift invariant; the sums stay small, so
// that "sum of squares minus squared sum" keeps ~15 digits).
//
// Gaussian smoothing = scipy.ndimage.gaussian_filter defaults: separable, axis 0 then 1 then 2, float64, kernel
// radius int(4 sigma + 0.5), 'reflect' boundary (d c b a | a b c d | d c b a).
#include "b4d_common.cuh"

namespace {

constexpr int COH_NSUM = 23;

__device__ __forceinline__ int reflect_idx(int i, int n) {
    // scipy 'reflect' (half-sample symmetric), any distance
    if (n == 1) return 0;
    const int period = 2 * n;
    i %= period;
    if (i < 0) i += period;
    return i < n ? i : period - 1 - i;
}

// centred float64 copy: x = raw - raw[first voxel of the patch]
__global__ void __launch_bounds__(256) k_coh_centre(const float *__restrict__ raw, double *__restrict__ x, long long V,
                                                    long long npatch) {
    const long long total = V * npatch, stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long p = i / V;
        x[i] = (double)raw[i] - (double)__ldg(raw + p * V);
    }
}

// one separable pass of the Gaussian filter along `axis` (0 = z, 1 = y, 2 = x)
__global__ void __launch_bounds__(256) k_coh_gauss(const double *__restrict__ in, double *__restrict__ out, int D, int H,
                                                   int W, long long npatch, int axis, int radius, const double *__restrict__ w) {
    const long long V = (long long)D * H * W, total = V * npatch, stride = (long long)gridDim.x * blockDim.x;
    const int n = axis == 0 ? D : (axis == 1 ? H : W);
    const long long step = axis == 0 ? (long long)H * W : (axis == 1 ? W : 1);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long v = i % V;
        const int c = axis == 0 ? (int)(v / ((long long)H * W)) : (axis == 1 ? (int)((v / W) % H) : (int)(v % W));
        const double *line = in + (i - (long long)c * step);
        double acc = 0.0;
        for (int k = -radius; k <= radius; ++k) acc = fma(w[k + radius], line[(long long)reflect_idx(c + k, n) * step], acc);
        out[i] = acc;
    }
}

// ---- label table: open addressing on the 64-bit label id, one table of `cap` slots per patch -------------
__device__ __forceinline__ uint32_t hash64(unsigned long long k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return (uint32_t)k;
}
// returns the slot of `key` (inserting it), or -1 when the table is full
__device__ __forceinline__ int table_slot(unsigned long long *keys, int cap, unsigned long long key, bool insert) {
    uint32_t s = hash64(key) & (uint32_t)(cap - 1);
    for (int probe = 0; probe < cap; ++probe) {
        const unsigned long long cur = keys[s];
        if (cur == key) return (int)s;
        if (cur == 0ull) {
            if (!insert) return -1;
            const unsigned long long old = atomicCAS(keys + s, 0ull, key);
            if (old == 0ull || old == key) return (int)s;
        }
        s = (s + 1) & (uint32_t)(cap - 1);
    }
    return -1;
}
__global__ void __launch_bounds__(256) k_coh_labels(const unsigned long long *__restrict__ labels, long long V,
                                                    long long npatch, unsigned long long *__restrict__ keys, int cap,
                                                    int *__restrict__ overflow) {
    const long long total = V * npatch, stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const unsigned long long l = labels[i];
        if (l == 0ull) continue;
        const unsigned long long prev = (i % V) ? labels[i - 1] : 0ull;
        if (prev == l) continue;  // runs along x: one insertion per run
        if (table_slot(keys + (i / V) * cap, cap, l, true) < 0) atomicExch(overflow, 1);
    }
}

// ---- the 23 sums per (patch, slot).  A warp covers 32 consecutive voxels; lanes that share a slot are summed by
// the lowest lane of their group before one double atomic per sum goes to memory.
__global__ void __launch_bounds__(256) k_coh_sums(const double *__restrict__ x, const double *__restrict__ sm,
                                                  const unsigned long long *__restrict__ labels, int D, int H, int W,
                                                  long long npatch, int lag, const unsigned long long *__restrict__ keys,
                                                  int cap, double *__restrict__ sums) {
    const long long V = (long long)D * H * W, total = V * npatch;
    const long long nwarp_total = (total + 31) / 32;
    const int lane = threadIdx.x & 31;
    const long long wstride = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long wi = (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5); wi < nwarp_total; wi += wstride) {
        const long long i = wi * 32 + lane;
        int slot = -1;
        double val[COH_NSUM];
#pragma unroll
        for (int q = 0; q < COH_NSUM; ++q) val[q] = 0.0;
        long long p = 0;
        if (i < total) {
            p = i / V;
            const unsigned long long l = labels[i];
            if (l != 0ull) {
                slot = table_slot(const_cast<unsigned long long *>(keys) + p * cap, cap, l, false);
                const long long v = i - p * V;
                const int cz = (int)(v / ((long long)H * W)), cy = (int)((v / W) % H), cx = (int)(v % W);
                const double xv = x[i], hv = xv - sm[i];
                val[0] = 1.0;
                val[1] = xv;
                val[2] = xv * xv;
                val[3] = hv;
                val[4] = hv * hv;
                const int c[3] = {cz, cy, cx}, n[3] = {D, H, W};
                const long long st[3] = {(long long)H * W, W, 1};
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    if (c[a] + lag < n[a] && labels[i + lag * st[a]] == l) {  // pair (this voxel, +lag) inside the segment
                        const double yv = x[i + lag * st[a]];
                        val[5 + 6 * a + 0] = 1.0;
                        val[5 + 6 * a + 1] = xv;
                        val[5 + 6 * a + 2] = yv;
                        val[5 + 6 * a + 3] = xv * xv;
                        val[5 + 6 * a + 4] = yv * yv;
                        val[5 + 6 * a + 5] = xv * yv;
                    }
                }
            }
        }
        // group lanes by (patch, slot); patch changes at most once inside a warp
        const long long gkey = slot < 0 ? -1 : p * cap + slot;
        const unsigned peers = __match_any_sync(B4D_FULL, gkey);
        const int leader = __ffs(peers) - 1;
        if (peers == B4D_FULL) {  // the common case: one segment (or background) across the warp
            if (gkey >= 0) {
#pragma unroll
                for (int q = 0; q < COH_NSUM; ++q) {
                    double s = val[q];
#pragma unroll
                    for (int m = 16; m >= 1; m >>= 1) s += __shfl_xor_sync(B4D_FULL, s, m);
                    if (lane == 0 && s != 0.0) atomicAdd(sums + gkey * COH_NSUM + q, s);
                }
            }
        } else {
            // mixed warp: every group's leader gathers its members' values lane by lane
#pragma unroll
            for (int q = 0; q < COH_NSUM; ++q) {
                double s = 0.0;
#pragma unroll 4
                for (int src = 0; src < 32; ++src) {
                    const double o = __shfl_sync(B4D_FULL, val[q], src);
                    if ((peers >> src) & 1u) s += o;
                }
                if (lane == leader && gkey >= 0 && s != 0.0) atomicAdd(sums + gkey * COH_NSUM + q, s);
            }
        }
    }
}

unsigned grid_of(long long n) {
    long long b = (n + 255) / 256;
    return (unsigned)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));
}

}  // namespace

// raw [npatch][D][H][W] float32, labels uint64 (0 = background); x, sm, tmp: float64 scratch of the same element
// count; keys [npatch][cap] (zeroed here), sums [npatch][cap][23] (zeroed here); w: device copy of the 2 radius + 1
// Gaussian weights; overflow: device int, set when a patch holds more distinct labels than the table takes.
void b4d_launch_coherence(const float *raw, const unsigned long long *labels, int D, int H, int W, long long npatch,
                          int lag, int radius, const double *w, double *x, double *sm, double *tmp,
                          unsigned long long *keys, int cap, double *sums, int *overflow, cudaStream_t s) {
    const long long V = (long long)D * H * W, total = V * npatch;
    cudaMemsetAsync(keys, 0, (size_t)npatch * cap * sizeof(unsigned long long), s);
    cudaMemsetAsync(sums, 0, (size_t)npatch * cap * COH_NSUM * sizeof(double), s);
    cudaMemsetAsync(overflow, 0, sizeof(int), s);
    b4d_launch(k_coh_centre, grid_of(total), 256, 0, s, raw, x, V, npatch);
    b4d_launch(k_coh_gauss, grid_of(total), 256, 0, s, x, sm, D, H, W, npatch, 0, radius, w);
    b4d_launch(k_coh_gauss, grid_of(total), 256, 0, s, sm, tmp, D, H, W, npatch, 1, radius, w);
    b4d_launch(k_coh_gauss, grid_of(total), 256, 0, s, tmp, sm, D, H, W, npatch, 2, radius, w);
    b4d_launch(k_coh_labels, grid_of(total), 256, 0, s, labels, V, npatch, keys, cap, overflow);
    b4d_launch(k_coh_sums, grid_of(total), 256, 0, s, x, sm, labels, D, H, W, npatch, lag, keys, cap, sums);
}
