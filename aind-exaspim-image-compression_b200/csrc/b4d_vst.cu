// b4d_vst.cu — the generalized Anscombe transform of Poisson-Gaussian counts (DESIGN §3.12).
//
// Forward: uint16 z -> float32 f = 2 sqrt(max((z - mu)/alpha + 3/8 + q^2, 0)), q = sigma/alpha.  Inverse: the
// closed-form approximation of the exact unbiased inverse (Makitalo & Foi 2013), float32 D -> float32
// alpha lambda + mu, or, fused with K7, the uint16 value b4d_quantize_u16 / _trunc_u16 would give on it.
// Elementwise and float64 inside: every operation is one IEEE + - * / sqrt in the order of the contract (the
// build uses -fmad=false), so a NumPy float64 restatement in the same order is bit-exact.  Scalar accesses, so
// any pointer alignment works; a warp still reads and writes contiguous runs.
#include <algorithm>

#include "b4d_common.cuh"

namespace {

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
unsigned grid_for(long long n) {
    const long long want = std::max(1ll, (n + 255) / 256);
    return (unsigned)std::min<long long>(want, 8ll * sm_count());
}

__device__ __forceinline__ float gat_forward1(uint32_t z, const GatParams &p) {
    const double t = (((double)z - p.offset) / p.gain + 0.375) + p.qq;
    return (float)(2.0 * sqrt(t > 0.0 ? t : 0.0));
}

__global__ void __launch_bounds__(256) k_gat_forward(const uint16_t *__restrict__ in, float *__restrict__ out,
                                                     long long n, GatParams p) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        __stcs(out + i, gat_forward1(__ldcs(in + i), p));
}

// The value set of a VST pass: list[i] = f(vals[i]), table[vals[i]] = f(vals[i]).
__global__ void __launch_bounds__(256) k_gat_values(const uint16_t *__restrict__ vals, int m, GatParams p,
                                                    float *__restrict__ list, float *__restrict__ table) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
        const uint32_t u = vals[i];
        const float f = gat_forward1(u, p);
        list[i] = f;
        table[u] = f;
    }
}

// Forward with a known map: the float32 data and the matching image of a volume in one pass, from the 256 KB value
// table (L2- and L1-resident).  A NaN entry marks a value outside the value set.  in / match may alias: every
// thread reads its element before it writes it.
__global__ void __launch_bounds__(256) k_gat_forward_map(const uint16_t *in, const float *__restrict__ table,
                                                         float *__restrict__ zf, uint16_t *match, long long n,
                                                         float cf, float scale, int ishift, unsigned *absent) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    bool bad = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float v = __ldg(table + in[i]);
        bad |= isnan(v);
        __stcs(zf + i, v);
        match[i] = (uint16_t)to_match(v, cf, scale, ishift);
    }
    if (__any_sync(B4D_FULL, bad) && (threadIdx.x & 31) == 0) atomicOr(absent, 1u);
}

// Q: write K7 of the result (TRUNC: the truncating variant) into q16 instead of the float32 result into out.
// out may be in (in place).
template <bool Q, bool TRUNC>
__global__ void __launch_bounds__(256) k_gat_inverse(const float *in, float *out, uint16_t *q16, long long n, GatParams p,
                                                     float osub, float oadd, float step) {
    const bool unit = (step == 1.0f);
    const float hi = __fdiv_rn(65535.0f, step);  // as k_quantize
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float y = gat_inverse1(__ldcs(in + i), p);
        if (Q) q16[i] = (uint16_t)quantq<TRUNC>(y, osub, oadd, step, hi, unit);
        else out[i] = y;
    }
}

}  // namespace

void b4d_launch_gat_forward(const uint16_t *in, float *out, long long n, const GatParams &p, cudaStream_t s) {
    b4d_launch(k_gat_forward, grid_for(n), 256, 0, s, in, out, n, p);
}

void b4d_launch_gat_inverse(const float *in, float *out, uint16_t *q16, long long n, const GatParams &p,
                            float offset_sub, float offset_add, float step, int trunc, cudaStream_t s) {
    const unsigned g = grid_for(n);
    if (!q16) b4d_launch(k_gat_inverse<false, false>, g, 256, 0, s, in, out, q16, n, p, offset_sub, offset_add, step);
    else if (trunc)
        b4d_launch(k_gat_inverse<true, true>, g, 256, 0, s, in, out, q16, n, p, offset_sub, offset_add, step);
    else b4d_launch(k_gat_inverse<true, false>, g, 256, 0, s, in, out, q16, n, p, offset_sub, offset_add, step);
}

void b4d_launch_gat_values(const uint16_t *vals, int m, const GatParams &p, float *list, float *table, cudaStream_t s) {
    b4d_launch(k_gat_values, grid_for(m), 256, 0, s, vals, m, p, list, table);
}

void b4d_launch_gat_forward_map(const uint16_t *in, const float *table, float *zf, uint16_t *match, long long n,
                                float cf, float scale, int ishift, unsigned *absent, cudaStream_t s) {
    b4d_launch(k_gat_forward_map, grid_for(n), 256, 0, s, in, table, zf, match, n, cf, scale, ishift, absent);
}
