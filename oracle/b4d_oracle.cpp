// b4d_oracle.cpp — CPU ORACLE for the BM4D denoise path.  TEST INFRASTRUCTURE ONLY.
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
// reference legs may load this library.  The product (libb4d.so) never does.
//
// PARITY UNPINNED.  The reference calls the closed third-party wheel
// bm4d==4.2.5 (uv.lock:387-400; call sites data_handling.py:332, :926 and
// evaluate.py:202).  It is absent from /root/reference, from this image and
// from the GPU box, and no reference test holds a single BM4D output value,
// so this file restates the PUBLISHED algorithm (Maggioni, Katkovnik,
// Egiazarian, Foi, IEEE TIP 2013) under the contract of SURVEY.md Appendix A /
// DESIGN.md §3.  Steps that DO exist in the reference tree are followed line
// by line in oracle/np_oracle.py and pinned against the imported reference
// (tests/golden/).
//
// Two independent arithmetic paths are provided on purpose:
//
//   arith = "f64"    plain restatement: dense orthonormal matrices (Haar-4 =
//                    periodised bior1.5 at L = 4, DCT-II-4, Haar-K), float64
//                    everywhere, float64 accumulators.  This is the oracle the
//                    tolerance test (max-abs 0.5, rel-L2 1e-3) is stated against.
//   arith = "mirror" the same algorithm in float32 with the operation order the
//                    CUDA kernels use (unnormalised butterflies, power-of-two
//                    rescale, fixed-point int64 aggregation).  With the
//                    profile's deterministic flag the CUDA path must equal this
//                    BIT FOR BIT — a much sharper regression check.
//
// Compile with -ffp-contract=off (oracle/Makefile does): the mirror path relies
// on every float operation being rounded exactly once, and uses fmaf() where
// the kernels use an explicit FMA.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <omp.h>

#include "../include/b4d.h"

namespace {

thread_local std::string g_err;
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

constexpr int L = 4;
constexpr int LV = 64;

struct b4d_handle_impl {
    b4d_profile prof;
    int arith;  // 0 = mirror (float32, CUDA op order), 1 = f64 plain restatement
    int threads;
    bool psd = false;  // coloured-noise model (b4d_set_noise_model)
    float nu_ht[64], nu_wie[64];
    mutable std::vector<int64_t> last_numq, last_wmap;  // mirror: accumulators of the last filter stage
    mutable std::vector<uint16_t> last_widx2;           // stage-2 match lists of the last two-stage call
    mutable std::vector<uint8_t> last_cnt2;
};

// ---------------------------------------------------------------- profile ---
void default_profile(b4d_profile *p) {
    std::memset(p, 0, sizeof(*p));
    p->abi = B4D_ABI_VERSION;
    p->block = 4;
    p->step = 3;
    p->search_ht = 11;
    p->search_wie = 11;
    p->k_ht = 16;
    p->k_wie = 32;
    p->stages = 2;
    p->deterministic = 0;
    p->tau_ht = 2.9527f;
    p->tau_wie = 0.7693f;
    p->lambda_ht = 2.7f;
    p->kaiser_beta = 2.0f;
}

bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

int check_profile(const b4d_profile &p) {
    if (p.abi != B4D_ABI_VERSION) return fail(B4D_ERR_INVALID, "profile.abi mismatch");
    if (p.block != 4 || p.step != 3)
        return fail(B4D_ERR_UNSUPPORTED, "only block = 4, step = 3 are implemented");
    for (int ns : {p.search_ht, p.search_wie})
        if (ns < 3 || ns > 15 || (ns & 1) == 0)
            return fail(B4D_ERR_INVALID, "search window side must be odd in [3, 15]");
    for (int k : {p.k_ht, p.k_wie})
        if (!is_pow2(k) || k > 32) return fail(B4D_ERR_INVALID, "group size must be a power of two <= 32");
    if (p.stages != 1 && p.stages != 2) return fail(B4D_ERR_INVALID, "stages must be 1 or 2");
    if (!(p.tau_ht > 0) || !(p.tau_wie > 0) || !(p.lambda_ht >= 0))
        return fail(B4D_ERR_INVALID, "tau / lambda must be positive");
    return 0;
}

// ------------------------------------------------------------------- grid ---
// Reference-block origins along one axis: 0, 3, 6, ... plus a final flush
// origin N - L when (N - L) is not on the grid (SURVEY Appendix A).
std::vector<int> ref_origins(int64_t n) {
    std::vector<int> o;
    for (int64_t v = 0; v + L <= n; v += 3) o.push_back((int)v);
    if ((n - L) % 3 != 0) o.push_back((int)(n - L));
    return o;
}

// z origins of one slab: global grid, kept when the whole search window lies
// inside the slab; returned in slab-local coordinates.
std::vector<int> slab_origins(int64_t z_total, int64_t z_begin, int64_t depth, int r) {
    std::vector<int> o;
    for (int g : ref_origins(z_total)) {
        int64_t lo = std::max<int64_t>(0, g - r);
        int64_t hi = std::min<int64_t>(z_total - L, g + r) + (L - 1);
        if (lo >= z_begin && hi < z_begin + depth) o.push_back((int)(g - z_begin));
    }
    return o;
}

struct Geom {
    int D, H, W;
    std::vector<int> rz, ry, rx;
    int64_t nrefs() const { return (int64_t)rz.size() * ry.size() * rx.size(); }
};

// -------------------------------------------------------------- matching ---
// Exact integer SSD over 4x4x4 blocks of a uint16 image; candidates are every
// origin of the Ns^3 window clipped to [0, N - L]; accepted when SSD <= tau;
// ordered by (SSD, window index (dz*Ns + dy)*Ns + dx); truncated to the largest
// power of two <= min(K, accepted).
struct Matches {
    int K;
    std::vector<uint16_t> widx;  // [R*K] window index
    std::vector<uint64_t> ssd;   // [R*K]
    std::vector<uint8_t> cnt;    // [R]
};

void match_all(const uint16_t *u, const Geom &g, int Ns, int K, uint64_t tau, Matches &m) {
    const int r = Ns / 2;
    const int64_t R = g.nrefs();
    m.K = K;
    m.widx.assign(R * K, 0xFFFF);
    m.ssd.assign(R * K, UINT64_MAX);
    m.cnt.assign(R, 0);
    const int nry = (int)g.ry.size(), nrx = (int)g.rx.size();
    const int64_t sy = g.W, sz = (int64_t)g.W * g.H;
#pragma omp parallel
    {
        std::vector<std::pair<uint64_t, uint32_t>> acc;
        acc.reserve(Ns * Ns * Ns);
#pragma omp for schedule(dynamic, 16)
        for (int64_t ri = 0; ri < R; ++ri) {
            const int oz = g.rz[ri / ((int64_t)nry * nrx)];
            const int oy = g.ry[(ri / nrx) % nry];
            const int ox = g.rx[ri % nrx];
            int32_t ref[LV];
            for (int z = 0; z < L; ++z)
                for (int y = 0; y < L; ++y)
                    for (int x = 0; x < L; ++x)
                        ref[(z * L + y) * L + x] = u[(oz + z) * sz + (oy + y) * sy + ox + x];
            acc.clear();
            const int z0 = std::max(0, oz - r), z1 = std::min(g.D - L, oz + r);
            const int y0 = std::max(0, oy - r), y1 = std::min(g.H - L, oy + r);
            const int x0 = std::max(0, ox - r), x1 = std::min(g.W - L, ox + r);
            for (int cz = z0; cz <= z1; ++cz)
                for (int cy = y0; cy <= y1; ++cy)
                    for (int cx = x0; cx <= x1; ++cx) {
                        uint64_t s = 0;
                        const uint16_t *c = u + cz * sz + cy * sy + cx;
                        for (int z = 0; z < L; ++z)
                            for (int y = 0; y < L; ++y) {
                                const uint16_t *row = c + z * sz + y * sy;
                                const int32_t *rr = ref + (z * L + y) * L;
                                for (int x = 0; x < L; ++x) {
                                    int64_t d = (int64_t)row[x] - rr[x];
                                    s += (uint64_t)(d * d);
                                }
                            }
                        if (s <= tau) {
                            uint32_t wi = (uint32_t)(((cz - (oz - r)) * Ns + (cy - (oy - r))) * Ns +
                                                     (cx - (ox - r)));
                            acc.emplace_back(s, wi);
                        }
                    }
            std::sort(acc.begin(), acc.end());
            int n = (int)std::min<size_t>(acc.size(), (size_t)K);
            int kp = 1;
            while (kp * 2 <= n) kp *= 2;
            if (n == 0) kp = 0;  // cannot happen: the reference block matches itself with SSD 0
            m.cnt[ri] = (uint8_t)kp;
            for (int k = 0; k < kp; ++k) {
                m.ssd[ri * K + k] = acc[k].first;
                m.widx[ri * K + k] = (uint16_t)acc[k].second;
            }
        }
    }
}

inline void widx_to_origin(int wi, int Ns, int r, int oz, int oy, int ox, int &cz, int &cy, int &cx) {
    cz = oz - r + wi / (Ns * Ns);
    cy = oy - r + (wi / Ns) % Ns;
    cx = ox - r + wi % Ns;
}

// ---------------------------------------------------------------- window ---
double bessel_i0(double x) {
    double s = 1.0, t = 1.0;
    for (int k = 1; k < 64; ++k) {
        t *= (x / (2.0 * k)) * (x / (2.0 * k));
        s += t;
        if (t < 1e-18 * s) break;
    }
    return s;
}
void kaiser4(double beta, double w[4]) {
    for (int n = 0; n < 4; ++n) {
        if (beta <= 0) {
            w[n] = 1.0;
            continue;
        }
        double a = 2.0 * n / 3.0 - 1.0;
        w[n] = bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - a * a))) / bessel_i0(beta);
    }
}

// =====================================================================
//  Path 1: plain float64 restatement with dense orthonormal matrices
// =====================================================================
struct Mats {
    double haar4[4][4], dct4[4][4];
};
Mats make_mats() {
    Mats m{};
    const double h = 0.5, q = 1.0 / std::sqrt(2.0);
    // Periodised bior1.5 analysis matrix at length 4, full decomposition,
    // row-normalised, equals the orthonormal Haar matrix (SURVEY §0.6).
    const double hh[4][4] = {{h, h, h, h}, {h, h, -h, -h}, {q, -q, 0, 0}, {0, 0, q, -q}};
    std::memcpy(m.haar4, hh, sizeof(hh));
    for (int k = 0; k < 4; ++k)
        for (int n = 0; n < 4; ++n) {
            double c = (k == 0) ? 0.5 : std::sqrt(0.5);
            m.dct4[k][n] = c * std::cos(M_PI * (2 * n + 1) * k / 8.0);
        }
    return m;
}
// Orthonormal Haar matrix of size K (power of two), full dyadic decomposition.
// Row layout: row 0 = scaling function; the detail of level l (l = 1 finest)
// covering samples [i, i + 2^l) sits at row i + 2^(l-1) — the same placement the
// in-place butterflies of the mirror path produce.
std::vector<double> haar_matrix(int K) {
    std::vector<double> m((size_t)K * K, 0.0);
    for (int j = 0; j < K; ++j) m[j] = 1.0 / std::sqrt((double)K);
    for (int s = 1; s < K; s *= 2)
        for (int i = 0; i < K; i += 2 * s) {
            double a = 1.0 / std::sqrt(2.0 * s);
            for (int j = 0; j < s; ++j) {
                m[(size_t)(i + s) * K + i + j] = a;
                m[(size_t)(i + s) * K + i + s + j] = -a;
            }
        }
    return m;
}

void sep3(const double T[4][4], bool transpose, const double *in, double *out) {
    double a[LV], b[LV];
    auto t = [&](int k, int n) { return transpose ? T[n][k] : T[k][n]; };
    for (int z = 0; z < 4; ++z)
        for (int y = 0; y < 4; ++y)
            for (int k = 0; k < 4; ++k) {
                double s = 0;
                for (int n = 0; n < 4; ++n) s += t(k, n) * in[(z * 4 + y) * 4 + n];
                a[(z * 4 + y) * 4 + k] = s;
            }
    for (int z = 0; z < 4; ++z)
        for (int x = 0; x < 4; ++x)
            for (int k = 0; k < 4; ++k) {
                double s = 0;
                for (int n = 0; n < 4; ++n) s += t(k, n) * a[(z * 4 + n) * 4 + x];
                b[(z * 4 + k) * 4 + x] = s;
            }
    for (int y = 0; y < 4; ++y)
        for (int x = 0; x < 4; ++x)
            for (int k = 0; k < 4; ++k) {
                double s = 0;
                for (int n = 0; n < 4; ++n) s += t(k, n) * b[(n * 4 + y) * 4 + x];
                out[(k * 4 + y) * 4 + x] = s;
            }
}

void group_xf(const std::vector<double> &G, int K, bool transpose, std::vector<double> &stack) {
    std::vector<double> tmp((size_t)K * LV);
    for (int k = 0; k < K; ++k)
        for (int v = 0; v < LV; ++v) {
            double s = 0;
            for (int j = 0; j < K; ++j)
                s += (transpose ? G[(size_t)j * K + k] : G[(size_t)k * K + j]) * stack[(size_t)j * LV + v];
            tmp[(size_t)k * LV + v] = s;
        }
    stack.swap(tmp);
}

template <bool WIENER>
void filter_f64(const float *zf, const double *basic, const Geom &g, const Matches &m, int Ns,
                double sigma, const b4d_profile &p, std::vector<double> &num,
                std::vector<double> &den, const float *nu = nullptr) {
    const Mats mats = make_mats();
    const int r = Ns / 2;
    double kw[4], win[LV];
    kaiser4(p.kaiser_beta, kw);
    for (int z = 0; z < 4; ++z)
        for (int y = 0; y < 4; ++y)
            for (int x = 0; x < 4; ++x) win[(z * 4 + y) * 4 + x] = kw[z] * kw[y] * kw[x];
    std::vector<std::vector<double>> hm(6);
    for (int l = 0; l <= 5; ++l) hm[l] = haar_matrix(1 << l);
    const int nry = (int)g.ry.size(), nrx = (int)g.rx.size();
    const int64_t sy = g.W, sz = (int64_t)g.W * g.H;
    const int64_t R = g.nrefs();
    const double thr = (double)p.lambda_ht * sigma;
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t ri = 0; ri < R; ++ri) {
        const int kp = m.cnt[ri];
        if (kp == 0) continue;
        int lg = 0;
        while ((1 << lg) < kp) ++lg;
        const int oz = g.rz[ri / ((int64_t)nry * nrx)];
        const int oy = g.ry[(ri / nrx) % nry];
        const int ox = g.rx[ri % nrx];
        int cz[32], cy[32], cx[32];
        std::vector<double> noisy((size_t)kp * LV), est((size_t)kp * LV);
        double blk[LV];
        for (int k = 0; k < kp; ++k) {
            widx_to_origin(m.widx[ri * m.K + k], Ns, r, oz, oy, ox, cz[k], cy[k], cx[k]);
            for (int z = 0; z < 4; ++z)
                for (int y = 0; y < 4; ++y)
                    for (int x = 0; x < 4; ++x)
                        blk[(z * 4 + y) * 4 + x] = zf[(cz[k] + z) * sz + (cy[k] + y) * sy + cx[k] + x];
            sep3(WIENER ? mats.dct4 : mats.haar4, false, blk, &noisy[(size_t)k * LV]);
            if (WIENER) {
                for (int z = 0; z < 4; ++z)
                    for (int y = 0; y < 4; ++y)
                        for (int x = 0; x < 4; ++x)
                            blk[(z * 4 + y) * 4 + x] =
                                basic[(cz[k] + z) * sz + (cy[k] + y) * sy + cx[k] + x];
                sep3(mats.dct4, false, blk, &est[(size_t)k * LV]);
            }
        }
        group_xf(hm[lg], kp, false, noisy);
        double weight;
        // coloured noise: coefficient v of every block has the variance sigma^2 nu[v] (nu = 1: white)
        if (!WIENER) {
            double kept = 0;
            for (size_t i = 0; i < noisy.size(); ++i) {
                const double nv = nu ? (double)nu[i % LV] : 1.0;
                if (std::fabs(noisy[i]) < thr * std::sqrt(nv))
                    noisy[i] = 0.0;
                else
                    kept += nv;
            }
            weight = 1.0 / std::max(kept, 1.0);  // sigma^-2 cancels in num/den
        } else {
            group_xf(hm[lg], kp, false, est);
            double sw2 = 0;
            for (size_t i = 0; i < noisy.size(); ++i) {
                const double nv = nu ? (double)nu[i % LV] : 1.0;
                double y2 = est[i] * est[i];
                double w = y2 / (y2 + sigma * sigma * nv);
                noisy[i] *= w;
                sw2 += w * w * nv;
            }
            weight = 1.0 / std::max(sw2, 1.0);
        }
        group_xf(hm[lg], kp, true, noisy);
        for (int k = 0; k < kp; ++k) {
            sep3(WIENER ? mats.dct4 : mats.haar4, true, &noisy[(size_t)k * LV], blk);
            for (int z = 0; z < 4; ++z)
                for (int y = 0; y < 4; ++y)
                    for (int x = 0; x < 4; ++x) {
                        const int v = (z * 4 + y) * 4 + x;
                        const int64_t a = (cz[k] + z) * sz + (cy[k] + y) * sy + cx[k] + x;
                        const double ww = weight * win[v];
#pragma omp atomic
                        num[a] += ww * blk[v];
#pragma omp atomic
                        den[a] += ww;
                    }
        }
    }
}

// =====================================================================
//  Path 2: float32 mirror of the CUDA kernels' operation order
// =====================================================================
struct MirrorTables {
    float win[LV];       // (w[z]*w[y])*w[x] in float32
    float kf[4];         // the per-axis factors w[n] (float32): the denominator convolves with them separably
    float tht[16];       // tht[m] = float(lambda*sigma*2^(m/2)), m = 6 - n + l
    // Wiener stage, unnormalised DCT butterflies: a raw coefficient with n odd positions (of x, y, z) at group
    // level l has the true value raw * S_n * 2^(-l/2), S_n = (1/2)^(3-n) c3^n, c3 = cos(3 pi/8)/sqrt 2
    float wa[24];        // [n][l] = float(S_n 2^(-l/2))
    float wb[24];        // [n][l] = float(S_n^2 2^(-l))
    float tq;            // float(1 + sqrt 2) = c1 / c3
    float sigma2;        // float(sigma)*float(sigma)
    // coloured noise: relative coefficient variances and the tables derived from them (csrc/b4d_api.cu make_tables)
    bool psd;
    float nu_ht[LV], nu_wie[LV], s2c[LV], thc[LV * 6];
};
MirrorTables make_tables(const b4d_profile &p, float sigma, const float *nu_ht = nullptr, const float *nu_wie = nullptr) {
    MirrorTables t{};
    t.psd = nu_ht != nullptr;
    for (int c = 0; c < 64; ++c) {
        t.nu_ht[c] = nu_ht ? nu_ht[c] : 1.0f;
        t.nu_wie[c] = nu_wie ? nu_wie[c] : 1.0f;
        {
            volatile float s2f = sigma * sigma;       // float32 product, as sigma2 below
            volatile float s2c = s2f * t.nu_wie[c];   // nu = 1 reproduces the white path bit for bit
            t.s2c[c] = s2c;
        }
        const int n = ((c & 3) >= 2) + (((c >> 2) & 3) >= 2) + ((c >> 4) >= 2);
        for (int l = 0; l < 6; ++l) {
            const int m = 6 - n + l;
            const double sc = std::ldexp(1.0, m / 2) * ((m & 1) ? M_SQRT2 : 1.0);
            t.thc[c * 6 + l] = (float)((double)p.lambda_ht * (double)sigma * sc * std::sqrt((double)t.nu_ht[c]));
        }
    }
    double kw[4];
    kaiser4(p.kaiser_beta, kw);
    float kf[4];
    for (int i = 0; i < 4; ++i) kf[i] = (float)kw[i];
    for (int i = 0; i < 4; ++i) t.kf[i] = kf[i];
    for (int z = 0; z < 4; ++z)
        for (int y = 0; y < 4; ++y)
            for (int x = 0; x < 4; ++x) t.win[(z * 4 + y) * 4 + x] = (kf[z] * kf[y]) * kf[x];
    for (int m = 0; m < 16; ++m) {
        double s = std::ldexp(1.0, m / 2) * ((m & 1) ? M_SQRT2 : 1.0);
        t.tht[m] = (float)((double)p.lambda_ht * (double)sigma * s);
    }
    const double c3 = std::cos(3.0 * M_PI / 8.0) * M_SQRT1_2;
    for (int n = 0; n < 4; ++n)
        for (int l = 0; l < 6; ++l) {
            const double sn = std::ldexp(1.0, -(3 - n)) * std::pow(c3, n);
            t.wa[n * 6 + l] = (float)(sn * std::ldexp(1.0, -(l / 2)) * ((l & 1) ? M_SQRT1_2 : 1.0));
            t.wb[n * 6 + l] = (float)(sn * sn * std::ldexp(1.0, -l));
        }
    t.tq = (float)(1.0 + M_SQRT2);
    t.sigma2 = sigma * sigma;
    return t;
}

// unnormalised Haar-4 butterflies, in place on 4 strided values
inline void haar4_fwd(float *v, int s) {
    float a = v[0] + v[s], b = v[2 * s] + v[3 * s], c = v[0] - v[s], d = v[2 * s] - v[3 * s];
    v[0] = a + b;
    v[s] = a - b;
    v[2 * s] = c;
    v[3 * s] = d;
}
inline void haar4_inv(float *v, int s) {
    float pp = v[0] + v[s], q = v[0] - v[s], y2 = v[2 * s], y3 = v[3 * s];
    v[0] = pp + y2;
    v[s] = pp - y2;
    v[2 * s] = q + y3;
    v[3 * s] = q - y3;
}
// DCT-II-4 in unnormalised even/odd form: X0 = a + b, X2 = a - b, X1 = t c + d, X3 = c - t d, t = 1 + sqrt 2;
// true values 1/2 X0, 1/2 X2, c3 X1, c3 X3.  The inverse expects coefficients pre-scaled by the same factors.
inline void dct4_fwd(float *v, int s, float tq) {
    float a = v[0] + v[3 * s], b = v[s] + v[2 * s], c = v[0] - v[3 * s], d = v[s] - v[2 * s];
    v[0] = a + b;
    v[2 * s] = a - b;
    v[s] = fmaf(tq, c, d);
    v[3 * s] = fmaf(-tq, d, c);
}
inline void dct4_inv(float *v, int s, float tq) {
    float a = v[0] + v[2 * s], b = v[0] - v[2 * s];
    float c = fmaf(tq, v[s], v[3 * s]), d = fmaf(-tq, v[3 * s], v[s]);
    v[0] = a + c;
    v[3 * s] = a - c;
    v[s] = b + d;
    v[2 * s] = b - d;
}
template <bool DCT>
inline void xf3_fwd(float *b, const MirrorTables &t) {
    for (int i = 0; i < 16; ++i) DCT ? dct4_fwd(b + 4 * i, 1, t.tq) : haar4_fwd(b + 4 * i, 1);
    for (int z = 0; z < 4; ++z)
        for (int x = 0; x < 4; ++x) DCT ? dct4_fwd(b + 16 * z + x, 4, t.tq) : haar4_fwd(b + 16 * z + x, 4);
    for (int i = 0; i < 16; ++i) DCT ? dct4_fwd(b + i, 16, t.tq) : haar4_fwd(b + i, 16);
}
template <bool DCT>
inline void xf3_inv(float *b, const MirrorTables &t) {
    for (int i = 0; i < 16; ++i) DCT ? dct4_inv(b + i, 16, t.tq) : haar4_inv(b + i, 16);
    for (int z = 0; z < 4; ++z)
        for (int x = 0; x < 4; ++x) DCT ? dct4_inv(b + 16 * z + x, 4, t.tq) : haar4_inv(b + 16 * z + x, 4);
    for (int i = 0; i < 16; ++i) DCT ? dct4_inv(b + 4 * i, 1, t.tq) : haar4_inv(b + 4 * i, 1);
}
// in-place unnormalised Haar along the group, element k of block-major stack
inline void ghaar_fwd(float *st, int kp) {
    for (int s = 1; s < kp; s *= 2)
        for (int i = 0; i < kp; i += 2 * s)
            for (int v = 0; v < LV; ++v) {
                float a = st[i * LV + v], b = st[(i + s) * LV + v];
                st[i * LV + v] = a + b;
                st[(i + s) * LV + v] = a - b;
            }
}
inline void ghaar_inv(float *st, int kp) {
    for (int s = kp / 2; s >= 1; s /= 2)
        for (int i = 0; i < kp; i += 2 * s)
            for (int v = 0; v < LV; ++v) {
                float a = st[i * LV + v], b = st[(i + s) * LV + v];
                st[i * LV + v] = a + b;
                st[(i + s) * LV + v] = a - b;
            }
}
// detail level of group slot k: l = 1 + log2(lowest set bit); slot 0 -> log2(kp)
inline int group_level(int k, int lg) { return k == 0 ? lg : 1 + __builtin_ctz((unsigned)k); }
inline int spatial_class(int v) { return ((v & 3) >= 2) + (((v >> 2) & 3) >= 2) + ((v >> 4) >= 2); }

// Aggregation in fixed point (order independent), as csrc/b4d_filter.cu does: the weight of a
// block position is quantised to 20 bits, wq = rint(w*win*2^20); the denominator is the integer
// sum of wq, the numerator the sum of rint(wq*qscale*x) clamped below 2^39 (qscale = the
// power-of-two scale of the matching map, so that |x|*qscale stays within the 16-bit range).
constexpr float W_SCALE = 1048576.0f;  // 2^20
constexpr float Q_LIMIT = 5.49e11f;    // < 2^39

// number of odd positions of a DCT coefficient index v = (z*4 + y)*4 + x: its scale class
inline int dct_class(int v) { return (v & 1) + ((v >> 2) & 1) + ((v >> 4) & 1); }

template <bool WIENER>
void filter_mirror(const float *zf, const float *basic, const Geom &g, const Matches &m, int Ns,
                   const MirrorTables &t, float qscale, std::vector<int64_t> &numq, std::vector<int64_t> &denq) {
    const int r = Ns / 2;
    const int nry = (int)g.ry.size(), nrx = (int)g.rx.size();
    const int64_t sy = g.W, sz = (int64_t)g.W * g.H;
    const int64_t R = g.nrefs();
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t ri = 0; ri < R; ++ri) {
        const int kp = m.cnt[ri];
        if (kp == 0) continue;
        int lg = 0;
        while ((1 << lg) < kp) ++lg;
        const int oz = g.rz[ri / ((int64_t)nry * nrx)];
        const int oy = g.ry[(ri / nrx) % nry];
        const int ox = g.rx[ri % nrx];
        int cz[32], cy[32], cx[32];
        float noisy[32 * LV], est[32 * LV];
        for (int k = 0; k < kp; ++k) {
            widx_to_origin(m.widx[ri * m.K + k], Ns, r, oz, oy, ox, cz[k], cy[k], cx[k]);
            for (int z = 0; z < 4; ++z)
                for (int y = 0; y < 4; ++y)
                    for (int x = 0; x < 4; ++x) {
                        const int64_t a = (cz[k] + z) * sz + (cy[k] + y) * sy + cx[k] + x;
                        noisy[k * LV + (z * 4 + y) * 4 + x] = zf[a];
                        if (WIENER) est[k * LV + (z * 4 + y) * 4 + x] = basic[a];
                    }
        }
        // Operation order of csrc/b4d_filter.cu: Haar along the GROUP first (layout A of the kernel), then the
        // separable 3-D transform of every coefficient block (layout B), shrinkage, and back the same way.
        float weight;
        if (!WIENER) {
            ghaar_fwd(noisy, kp);
            for (int k = 0; k < kp; ++k) xf3_fwd<false>(noisy + k * LV, t);
            int kept = 0;
            float part[32];
            for (int k = 0; k < 32; ++k) part[k] = 0.0f;
            for (int k = 0; k < kp; ++k) {
                const int l = group_level(k, lg);
                // coloured noise: the weight sums nu_c of the retained coefficients in the kernel's order — lane k
                // chains (z, y, x pair (0|1) then (2|3)), low halves (x 0, 2) and high halves (x 1, 3) apart
                float kf_lo = 0.0f, kf_hi = 0.0f;
                for (int zy = 0; zy < 16; ++zy)
                    for (int o = 0; o < 2; ++o)
                        for (int hf = 0; hf < 2; ++hf) {
                            const int v = zy * 4 + 2 * o + hf;
                            const int n = spatial_class(v);
                            float c = noisy[k * LV + v];
                            const float th = t.psd ? t.thc[v * 6 + l] : t.tht[6 - n + l];
                            if (fabsf(c) < th) {
                                c = 0.0f;
                            } else {
                                ++kept;
                                (hf ? kf_hi : kf_lo) += t.nu_ht[v];
                                c = ldexpf(c, -(6 - n + l));  // exact: squared normalisation 2^(-6+n-l)
                            }
                            noisy[k * LV + v] = c;
                        }
                part[k] = kf_lo + kf_hi;
            }
            if (t.psd) {
                for (int mm = 16; mm >= 1; mm >>= 1) {
                    float nx[32];
                    for (int k = 0; k < 32; ++k) nx[k] = part[k] + part[k ^ mm];
                    std::memcpy(part, nx, sizeof(nx));
                }
                weight = 1.0f / fmaxf(part[0], 1.0f);
            } else {
                weight = 1.0f / (float)std::max(kept, 1);
            }
            for (int k = 0; k < kp; ++k) xf3_inv<false>(noisy + k * LV, t);
            ghaar_inv(noisy, kp);
        } else {
            ghaar_fwd(est, kp);
            for (int k = 0; k < kp; ++k) xf3_fwd<true>(est + k * LV, t);
            ghaar_fwd(noisy, kp);
            for (int k = 0; k < kp; ++k) xf3_fwd<true>(noisy + k * LV, t);
            const bool dump = getenv("B4D_DUMP_REF") && atoll(getenv("B4D_DUMP_REF")) == ri;  // developer aid
            auto dump_f = [&](int sec, const float *a) {
                for (int k = 0; k < kp; ++k)
                    for (int v = 0; v < LV; ++v) {
                        uint32_t b;
                        std::memcpy(&b, &a[k * LV + v], 4);
                        printf("D %d %d %d %08x\n", sec, k, v, b);
                    }
            };
            if (dump) {
                dump_f(0, est);
                dump_f(1, noisy);
            }
            // Wiener attenuation, elementwise.  Sum of W^2 in the kernel's order: lane k owns coefficient block
            // k and chains fma over its 64 coefficients as 32 packed pairs — for z, for y: the pair of x positions
            // (0, 2), then (1, 3) — low halves in one chain, high halves in the other; the two chains are added,
            // and the 32 lane sums meet in an xor butterfly (16, 8, 4, 2, 1).
            float part[32];
            for (int k = 0; k < 32; ++k) part[k] = 0.0f;
            for (int k = 0; k < kp; ++k) {
                const int l = group_level(k, lg);
                float acc_lo = 0.0f, acc_hi = 0.0f;
                for (int zy = 0; zy < 16; ++zy)
                    for (int o = 0; o < 2; ++o)
                        for (int h = 0; h < 2; ++h) {
                            const int v = zy * 4 + o + 2 * h;  // x position: (0 | 2) for o = 0, (1 | 3) for o = 1
                            const int n = dct_class(v);
                            const float yn = est[k * LV + v] * t.wa[n * 6 + l];
                            const float y2 = yn * yn;
                            const float nd = (t.psd ? -t.s2c[v] : -t.sigma2) - y2;
                            const float w = y2 / (-nd);
                            if (t.psd) {  // sum of W^2 nu_c as fma(W nu_c, W, acc): nu = 1 is the white chain
                                const float wn = w * t.nu_wie[v];
                                if (h == 0) acc_lo = fmaf(wn, w, acc_lo);
                                else acc_hi = fmaf(wn, w, acc_hi);
                            } else if (h == 0) {
                                acc_lo = fmaf(w, w, acc_lo);
                            } else {
                                acc_hi = fmaf(w, w, acc_hi);
                            }
                            noisy[k * LV + v] = (noisy[k * LV + v] * w) * t.wb[n * 6 + l];
                        }
                part[k] = acc_lo + acc_hi;
            }
            for (int mm = 16; mm >= 1; mm >>= 1) {  // xor-butterfly reduction, as __shfl_xor does
                float nx[32];
                for (int k = 0; k < 32; ++k) nx[k] = part[k] + part[k ^ mm];
                std::memcpy(part, nx, sizeof(nx));
            }
            weight = 1.0f / fmaxf(part[0], 1.0f);
            if (dump) dump_f(2, noisy);
            for (int k = 0; k < kp; ++k) xf3_inv<true>(noisy + k * LV, t);
            if (dump) dump_f(5, noisy);
            ghaar_inv(noisy, kp);
            if (dump) dump_f(3, noisy);
        }
        // Weight-map contract: the group weight is quantised once, qg = rint(w * 2^20); the numerator
        // term of a voxel uses the float32 weight float(qg) * win[v] (limb format as before), the
        // denominator is NOT accumulated per voxel: G[origin] += qg once per grouped block, and
        // den = G (*) window is evaluated by the normalise step (den_from_weight_map).
        const int64_t qg = (int64_t)lrintf(weight * W_SCALE);
        for (int k = 0; k < kp; ++k) {
#pragma omp atomic
            denq[cz[k] * sz + cy[k] * sy + cx[k]] += qg;
            for (int z = 0; z < 4; ++z)
                for (int y = 0; y < 4; ++y)
                    for (int x = 0; x < 4; ++x) {
                        const int v = (z * 4 + y) * 4 + x;
                        const int64_t a = (cz[k] + z) * sz + (cy[k] + y) * sy + cx[k] + x;
                        const float wqf = ((float)qg * t.win[v]) * qscale;
                        const float tq = fminf(fmaxf(wqf * noisy[k * LV + v], -Q_LIMIT), Q_LIMIT);
                        const int64_t qn = llrintf(tq);
                        if (WIENER && getenv("B4D_DUMP_REF") && atoll(getenv("B4D_DUMP_REF")) == ri) {
                            uint32_t b0, b1;
                            std::memcpy(&b0, &tq, 4);
                            std::memcpy(&b1, &wqf, 4);
                            printf("D 6 %d %d %08x\nD 7 %d %d %08x\n", k, v, b0, k, v, b1);
                        }
#pragma omp atomic
                        numq[a] += qn;
                    }
        }
    }
}

// den(v) = sum over block origins o = v - (dz, dy, dx), 0 <= d < 4, of G[o] * kf[dz] * kf[dy] * kf[dx]:
// three 4-tap passes (x, then y, then z) in float64, each an fma chain over d = 0..3 in that order —
// the order the normalise kernel has to follow.
void den_from_weight_map(const std::vector<int64_t> &G, const Geom &g, const MirrorTables &t, std::vector<double> &den) {
    const int D = g.D, H = g.H, W = g.W;
    const int64_t V = (int64_t)D * H * W;
    std::vector<double> a((size_t)V), b((size_t)V);
    const double k[4] = {(double)t.kf[0], (double)t.kf[1], (double)t.kf[2], (double)t.kf[3]};
#pragma omp parallel for
    for (int64_t zy = 0; zy < (int64_t)D * H; ++zy)
        for (int x = 0; x < W; ++x) {
            double acc = 0.0;
            for (int d = 0; d < 4 && d <= x; ++d) acc = std::fma(k[d], (double)G[zy * W + x - d], acc);
            a[zy * W + x] = acc;
        }
#pragma omp parallel for
    for (int z = 0; z < D; ++z)
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x) {
                double acc = 0.0;
                for (int d = 0; d < 4 && d <= y; ++d) acc = std::fma(k[d], a[((int64_t)z * H + y - d) * W + x], acc);
                b[((int64_t)z * H + y) * W + x] = acc;
            }
    den.assign((size_t)V, 0.0);
#pragma omp parallel for
    for (int z = 0; z < D; ++z)
        for (int64_t yx = 0; yx < (int64_t)H * W; ++yx) {
            double acc = 0.0;
            for (int d = 0; d < 4 && d <= z; ++d) acc = std::fma(k[d], b[(int64_t)(z - d) * H * W + yx], acc);
            den[(int64_t)z * H * W + yx] = acc;
        }
}

// ----------------------------------------------------- matching image ------
// Matching runs on a uint16 image:
//     u = clamp(int(rint((z + cf) * scale)) + ishift, 0, 65535)
//  * uint16 input: stage 1 matches on the data itself.
//  * float32 input that is uint16 counts minus one scalar (data_handling.py:
//    353-354): cf restores the integers (|cf| <= 0.5), scale 1 — matching is then
//    exactly the matching on the original counts (offset invariance).  "Counts" means
//    every value within min(1, sigma)/64 of an integer after the shift: data whose
//    whole range is that close to one integer only because sigma is small are not.
//  * any other float32 input: cf 0 and a power-of-two scale that puts sigma at
//    32..64 steps (bounded by the 16-bit range).
// Stage 2 quantises the basic estimate with cf = 0: u = int(rint(y*scale)) + ishift.
// ishift is an INTEGER that centres the range in uint16, applied after rounding,
// so the rounding never depends on it (a batch and a single patch agree).
struct MatchMap {
    float cf, scale;
    int ishift;
    int integral;
};
int centre_shift(double lo, double hi) { return (int)(std::floor((65535.0 - (hi - lo)) * 0.5) - lo); }
// *centre: see csrc/b4d_api.cu derive_match_map (large-DC float data are denoised on z - c0)
constexpr double CENTRE_LIMIT = 131072.0;
MatchMap derive_match_map(const float *z, int64_t n, float sigma, float *centre = nullptr) {
    double c = std::rint((double)z[0]) - (double)z[0];
    double dev = 0, lo = 1e300, hi = -1e300, zlo = 1e300, zhi = -1e300;
#pragma omp parallel for reduction(max : dev, hi, zhi) reduction(min : lo, zlo)
    for (int64_t i = 0; i < n; ++i) {
        double v = (double)z[i] + c, rv = std::rint(v);
        dev = std::max(dev, std::fabs(v - rv));
        lo = std::min(lo, rv);
        hi = std::max(hi, rv);
        zlo = std::min(zlo, (double)z[i]);
        zhi = std::max(zhi, (double)z[i]);
    }
    MatchMap mm{};
    if (dev <= std::min(1.0, (double)sigma) / 64.0 && hi - lo <= 65535.0) {
        mm.integral = 1;
        mm.scale = 1.0f;
        mm.cf = (float)c;
        mm.ishift = centre_shift(lo, hi);
    } else {
        double range = std::max(zhi - zlo, 1e-30);
        int e_range = (int)std::floor(std::log2(65535.0 / range));
        int e_sigma = (int)std::floor(std::log2(64.0 / (double)sigma));
        int e = std::min(e_range, e_sigma);
        mm.integral = 0;
        mm.scale = (float)std::ldexp(1.0, e);
        mm.cf = 0.0f;
        mm.ishift = centre_shift(std::floor(zlo * (double)mm.scale), std::ceil(zhi * (double)mm.scale));
    }
    if (centre) {
        const double peak = std::max(std::fabs(zlo), std::fabs(zhi)) * (double)mm.scale;
        *centre = 0.0f;
        if (peak > CENTRE_LIMIT) *centre = mm.integral ? (float)std::rint(0.5 * (lo + hi)) : (float)(0.5 * (zlo + zhi));
    }
    return mm;
}
inline uint16_t to_match_u16(float v, float cf, float scale, int ishift) {
    long long q = (long long)rintf((v + cf) * scale) + ishift;
    q = std::min<long long>(std::max<long long>(q, 0), 65535);
    return (uint16_t)q;
}

uint64_t tau_int(float tau, float sigma, float scale) {
    double s = (double)sigma * (double)scale;
    return (uint64_t)std::floor((double)tau * s * s * 64.0);
}

// ----------------------------------------------------------- full pipeline --
int denoise_one(const b4d_handle_impl *h, const uint16_t *in_u16, const float *in_f32, const Geom &g1,
                const Geom &g2, float sigma, float *out) {
    const b4d_profile &p = h->prof;
    const int64_t V = (int64_t)g1.D * g1.H * g1.W;
    std::vector<float> zf(V);
    std::vector<uint16_t> u(V);
    MatchMap mm{0.0f, 1.0f, 0, 1};
    if (in_u16) {
        // stage 1 matches on the raw integers; the stage-2 matching image is the
        // basic estimate centred in the uint16 range so that it is never clamped
        double lo = 65535.0, hi = 0.0;
        for (int64_t i = 0; i < V; ++i) {
            zf[i] = (float)in_u16[i];
            u[i] = in_u16[i];
            lo = std::min(lo, (double)in_u16[i]);
            hi = std::max(hi, (double)in_u16[i]);
        }
        mm.ishift = centre_shift(lo, hi);
    } else {
        for (int64_t i = 0; i < V; ++i)
            if (!std::isfinite(in_f32[i])) return fail(B4D_ERR_INVALID, "input contains non-finite values (NaN or infinity)");
        float centre = 0.0f;
        mm = derive_match_map(in_f32, V, sigma, &centre);
        if (centre != 0.0f) {  // large DC level: denoise z - c0, add c0 back (csrc/b4d_api.cu denoise_batch)
            std::vector<float> shifted(V);
            for (int64_t i = 0; i < V; ++i) shifted[i] = in_f32[i] + (-centre);
            if (int e = denoise_one(h, nullptr, shifted.data(), g1, g2, sigma, out)) return e;
            for (int64_t i = 0; i < V; ++i) out[i] = out[i] + centre;
            return 0;
        }
        for (int64_t i = 0; i < V; ++i) {
            zf[i] = in_f32[i];
            u[i] = to_match_u16(in_f32[i], mm.cf, mm.scale, mm.ishift);
        }
    }
    Matches m;
    match_all(u.data(), g1, p.search_ht, p.k_ht, tau_int(p.tau_ht, sigma, mm.scale), m);
    if (h->arith == 1) {
        std::vector<double> num(V, 0.0), den(V, 0.0), basic(V);
        filter_f64<false>(zf.data(), nullptr, g1, m, p.search_ht, (double)sigma, p, num, den, h->psd ? h->nu_ht : nullptr);
        for (int64_t i = 0; i < V; ++i) basic[i] = den[i] > 0 ? num[i] / den[i] : (double)zf[i];
        if (p.stages == 1) {
            for (int64_t i = 0; i < V; ++i) out[i] = (float)basic[i];
            return 0;
        }
        for (int64_t i = 0; i < V; ++i) u[i] = to_match_u16((float)basic[i], 0.0f, mm.scale, mm.ishift);
        match_all(u.data(), g2, p.search_wie, p.k_wie, tau_int(p.tau_wie, sigma, mm.scale), m);
        h->last_widx2 = m.widx;
        h->last_cnt2 = m.cnt;
        std::fill(num.begin(), num.end(), 0.0);
        std::fill(den.begin(), den.end(), 0.0);
        filter_f64<true>(zf.data(), basic.data(), g2, m, p.search_wie, (double)sigma, p, num, den,
                         h->psd ? h->nu_wie : nullptr);
        for (int64_t i = 0; i < V; ++i) out[i] = (float)(den[i] > 0 ? num[i] / den[i] : basic[i]);
        return 0;
    }
    const MirrorTables t = make_tables(p, sigma, h->psd ? h->nu_ht : nullptr, h->psd ? h->nu_wie : nullptr);
    std::vector<int64_t> numq(V, 0), denq(V, 0);
    std::vector<float> basic(V);
    const double inv_q = 1.0 / (double)mm.scale;
    std::vector<double> den;
    filter_mirror<false>(zf.data(), nullptr, g1, m, p.search_ht, t, mm.scale, numq, denq);
    den_from_weight_map(denq, g1, t, den);
    for (int64_t i = 0; i < V; ++i) basic[i] = den[i] > 0 ? (float)(((double)numq[i] / den[i]) * inv_q) : zf[i];
    h->last_numq = numq;
    h->last_wmap = denq;
    if (p.stages == 1) {
        std::memcpy(out, basic.data(), V * sizeof(float));
        return 0;
    }
    for (int64_t i = 0; i < V; ++i) u[i] = to_match_u16(basic[i], 0.0f, mm.scale, mm.ishift);
    match_all(u.data(), g2, p.search_wie, p.k_wie, tau_int(p.tau_wie, sigma, mm.scale), m);
    h->last_widx2 = m.widx;
    h->last_cnt2 = m.cnt;
    std::fill(numq.begin(), numq.end(), 0);
    std::fill(denq.begin(), denq.end(), 0);
    filter_mirror<true>(zf.data(), basic.data(), g2, m, p.search_wie, t, mm.scale, numq, denq);
    den_from_weight_map(denq, g2, t, den);
    for (int64_t i = 0; i < V; ++i) out[i] = den[i] > 0 ? (float)(((double)numq[i] / den[i]) * inv_q) : basic[i];
    h->last_numq = numq;
    h->last_wmap = denq;
    return 0;
}

int check_shape(const int64_t shape[3]) {
    for (int i = 0; i < 3; ++i)
        if (shape[i] < L || shape[i] > 65535)
            return fail(B4D_ERR_INVALID, "every dimension must be in [4, 65535]");
    return 0;
}
Geom whole_geom(const int64_t shape[3]) {
    Geom g;
    g.D = (int)shape[0];
    g.H = (int)shape[1];
    g.W = (int)shape[2];
    g.rz = ref_origins(shape[0]);
    g.ry = ref_origins(shape[1]);
    g.rx = ref_origins(shape[2]);
    return g;
}

}  // namespace

// =============================================================== C ABI =====
extern "C" {

int b4d_version(void) { return B4D_ABI_VERSION; }
const char *b4d_last_error(void) { return g_err.c_str(); }
void b4d_default_profile(b4d_profile *p) { default_profile(p); }

int b4d_create(int device, const b4d_profile *profile, b4d_handle **out) {
    (void)device;
    if (!out) return fail(B4D_ERR_INVALID, "out is NULL");
    auto *h = new b4d_handle_impl();
    default_profile(&h->prof);
    h->arith = 1;
    h->threads = 0;
    if (profile) {
        h->prof = *profile;
        if (int e = check_profile(h->prof)) {
            delete h;
            return e;
        }
    }
    *out = reinterpret_cast<b4d_handle *>(h);
    return 0;
}
void b4d_destroy(b4d_handle *h) { delete reinterpret_cast<b4d_handle_impl *>(h); }
int b4d_set_profile(b4d_handle *hh, const b4d_profile *profile) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || !profile) return fail(B4D_ERR_INVALID, "NULL argument");
    if (int e = check_profile(*profile)) return e;
    h->prof = *profile;
    return 0;
}
// oracle-only: choose the arithmetic path (0 = float32 mirror, 1 = float64 plain)
int b4d_oracle_set_arith(b4d_handle *hh, int arith) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || (arith != 0 && arith != 1)) return fail(B4D_ERR_INVALID, "arith must be 0 or 1");
    h->arith = arith;
    return 0;
}

// oracle-only: size of the OpenMP team (n <= 0 leaves it alone); returns the team size in effect.
// torch.distributed.run exports OMP_NUM_THREADS=1, so bench.py sets the count explicitly and reports this value.
int b4d_oracle_set_threads(int n) {
    if (n > 0) omp_set_num_threads(n);
    return omp_get_max_threads();
}

int64_t b4d_num_refs(const int64_t shape[3]) {
    if (check_shape(shape)) return -1;
    return whole_geom(shape).nrefs();
}

int b4d_denoise_u16(b4d_handle *hh, const uint16_t *in, int64_t n, const int64_t shape[3], float sigma,
                    float *out, int, int) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || !in || !out || n < 1) return fail(B4D_ERR_INVALID, "NULL argument or n < 1");
    if (!(sigma > 0)) return fail(B4D_ERR_INVALID, "sigma must be positive");
    if (int e = check_shape(shape)) return e;
    const Geom g = whole_geom(shape);
    const int64_t V = shape[0] * shape[1] * shape[2];
    for (int64_t i = 0; i < n; ++i)
        if (int e = denoise_one(h, in + i * V, nullptr, g, g, sigma, out + i * V)) return e;
    return 0;
}
int b4d_denoise_f32(b4d_handle *hh, const float *in, int64_t n, const int64_t shape[3], float sigma,
                    float *out, int, int) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || !in || !out || n < 1) return fail(B4D_ERR_INVALID, "NULL argument or n < 1");
    if (!(sigma > 0)) return fail(B4D_ERR_INVALID, "sigma must be positive");
    if (int e = check_shape(shape)) return e;
    const Geom g = whole_geom(shape);
    const int64_t V = shape[0] * shape[1] * shape[2];
    for (int64_t i = 0; i < n; ++i)
        if (int e = denoise_one(h, nullptr, in + i * V, g, g, sigma, out + i * V)) return e;
    return 0;
}

int b4d_denoise_slab_u16(b4d_handle *hh, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                         int64_t z_total, int64_t own_begin, int64_t own_end, float sigma, float *out,
                         int, int) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || !in || !out) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!(sigma > 0)) return fail(B4D_ERR_INVALID, "sigma must be positive");
    if (int e = check_shape(shape)) return e;
    if (z_begin < 0 || z_begin + shape[0] > z_total || own_begin < z_begin || own_end > z_begin + shape[0] ||
        own_begin >= own_end)
        return fail(B4D_ERR_INVALID, "slab / owned range inconsistent");
    Geom g1 = whole_geom(shape), g2 = g1;
    g1.rz = slab_origins(z_total, z_begin, shape[0], h->prof.search_ht / 2);
    g2.rz = slab_origins(z_total, z_begin, shape[0], h->prof.search_wie / 2);
    const int64_t V = shape[0] * shape[1] * shape[2], P = shape[1] * shape[2];
    std::vector<float> full(V);
    if (int e = denoise_one(h, in, nullptr, g1, g2, sigma, full.data())) return e;
    std::memcpy(out, full.data() + (own_begin - z_begin) * P, (own_end - own_begin) * P * sizeof(float));
    return 0;
}

int b4d_match_stage1(b4d_handle *hh, const uint16_t *in, const int64_t shape[3], float sigma, int32_t *idx,
                     uint64_t *ssd, int32_t *count) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || !in || !idx || !ssd || !count) return fail(B4D_ERR_INVALID, "NULL argument");
    if (int e = check_shape(shape)) return e;
    const Geom g = whole_geom(shape);
    const int64_t Hc = g.H - L + 1, Wc = g.W - L + 1, Dc = g.D - L + 1;
    if (Dc * Hc * Wc > INT32_MAX) return fail(B4D_ERR_TOO_LARGE, "candidate index space exceeds int32");
    const b4d_profile &p = h->prof;
    Matches m;
    match_all(in, g, p.search_ht, p.k_ht, tau_int(p.tau_ht, sigma, 1.0f), m);
    const int Ns = p.search_ht, r = Ns / 2, K = p.k_ht;
    const int nry = (int)g.ry.size(), nrx = (int)g.rx.size();
    const int64_t R = g.nrefs();
    for (int64_t ri = 0; ri < R; ++ri) {
        const int oz = g.rz[ri / ((int64_t)nry * nrx)], oy = g.ry[(ri / nrx) % nry], ox = g.rx[ri % nrx];
        count[ri] = m.cnt[ri];
        for (int k = 0; k < K; ++k) {
            if (k < m.cnt[ri]) {
                int cz, cy, cx;
                widx_to_origin(m.widx[ri * K + k], Ns, r, oz, oy, ox, cz, cy, cx);
                idx[ri * K + k] = (int32_t)(((int64_t)cz * Hc + cy) * Wc + cx);
                ssd[ri * K + k] = m.ssd[ri * K + k];
            } else {
                idx[ri * K + k] = -1;
                ssd[ri * K + k] = UINT64_MAX;
            }
        }
    }
    return 0;
}

// K7 restated in C (float32, clip before round, half-to-even): transforms.py:403-411.
int b4d_quantize_u16(b4d_handle *, const float *in, int64_t n, float offset_sub, float offset_add, float step,
                     uint16_t *out, int, int) {
    if (!in || !out || n < 0) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!(step >= 1.0f)) return fail(B4D_ERR_INVALID, "step must be >= 1");
    const float hi = 65535.0f / step;
    for (int64_t i = 0; i < n; ++i) {
        float v = (in[i] - offset_sub) + offset_add;
        if (step != 1.0f) v = v / step;
        v = fminf(fmaxf(v, 0.0f), hi);
        out[i] = (uint16_t)rintf(v);
    }
    return 0;
}

// truncating variant: np.maximum(x, 0).astype(int) (evaluate.py:202) + the uint16 cast of compute_cratio
// (utils/img_util.py:420-423): toward zero, no upper clip, int64 -> uint16 wraps modulo 2^16
int b4d_quantize_trunc_u16(b4d_handle *, const float *in, int64_t n, float offset_sub, float offset_add, float step,
                           uint16_t *out, int, int) {
    if (!in || !out || n < 0) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!(step >= 1.0f)) return fail(B4D_ERR_INVALID, "step must be >= 1");
    for (int64_t i = 0; i < n; ++i) {
        float v = (in[i] - offset_sub) + offset_add;
        if (step != 1.0f) v = v / step;
        v = std::isnan(v) ? 0.0f : fmaxf(v, 0.0f);
        out[i] = (uint16_t)((int64_t)v & 0xFFFF);
    }
    return 0;
}
// denoise -> quantize in one call: the restatement simply chains the two restated steps
int b4d_denoise_slab_q16_u16(b4d_handle *hh, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                             int64_t z_total, int64_t own_begin, int64_t own_end, float sigma, float offset_sub,
                             float offset_add, float step, int truncate, uint16_t *out, int, int) {
    if (!shape || !out || own_end <= own_begin) return fail(B4D_ERR_INVALID, "bad argument");
    const int64_t n = (own_end - own_begin) * shape[1] * shape[2];
    std::vector<float> y((size_t)n);
    if (int e = b4d_denoise_slab_u16(hh, in, shape, z_begin, z_total, own_begin, own_end, sigma, y.data(), 0, 0)) return e;
    return truncate ? b4d_quantize_trunc_u16(hh, y.data(), n, offset_sub, offset_add, step, out, 0, 0)
                    : b4d_quantize_u16(hh, y.data(), n, offset_sub, offset_add, step, out, 0, 0);
}
int b4d_denoise_q16_u16(b4d_handle *hh, const uint16_t *in, const int64_t shape[3], float sigma, float offset_sub,
                        float offset_add, float step, int truncate, uint16_t *out, int, int) {
    if (!shape) return fail(B4D_ERR_INVALID, "NULL argument");
    return b4d_denoise_slab_q16_u16(hh, in, shape, 0, shape[0], 0, shape[0], sigma, offset_sub, offset_add, step,
                                    truncate, out, 0, 0);
}
int b4d_slab_stage2_q16(b4d_handle *, int64_t, int64_t, float, float, float, int, uint16_t *, int) {
    return fail(B4D_ERR_UNSUPPORTED, "oracle: use b4d_denoise_slab_q16_u16");
}
int b4d_tile_stats(b4d_handle *, const uint16_t *, int64_t, double, b4d_stats *, int64_t *, int) {
    return fail(B4D_ERR_UNSUPPORTED, "tile statistics are restated in oracle/np_oracle.py (NumPy)");
}
int b4d_set_noise_model(b4d_handle *hh, const float *nu_ht, const float *nu_wie) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!nu_ht && !nu_wie) {
        h->psd = false;
        return 0;
    }
    if (!nu_ht || !nu_wie) return fail(B4D_ERR_INVALID, "both tables or none");
    std::memcpy(h->nu_ht, nu_ht, sizeof(h->nu_ht));
    std::memcpy(h->nu_wie, nu_wie, sizeof(h->nu_wie));
    h->psd = true;
    return 0;
}
int b4d_coherence_gate(b4d_handle *, const float *, const uint64_t *, int64_t, const int64_t *, double, double, int64_t,
                       double, int, uint8_t *, b4d_segment_score *, int64_t, int64_t *, int) {
    return fail(B4D_ERR_UNSUPPORTED, "the coherence gate is restated in oracle/np_oracle.py (NumPy / SciPy)");
}
int b4d_stats_from_hist(const int64_t *, double, b4d_stats *) {
    return fail(B4D_ERR_UNSUPPORTED, "tile statistics are restated in oracle/np_oracle.py (NumPy)");
}
void *b4d_stream(b4d_handle *) { return nullptr; }
int b4d_set_pass_voxels(b4d_handle *, int64_t) { return 0; }
int b4d_set_pipeline_min_voxels(b4d_handle *, int64_t) { return 0; }  // the CPU restatement has no passes
// restatement of make_foreground_mask (metrics.py:54-61) on raw = float32(u16) - offset
// (data_handling.py:353-354): plain float32 arrays, medians by selection, dilation by repeated
// 6-neighbour passes with border value 0 (scipy.ndimage.binary_dilation's default structure).
static float median_f32(std::vector<float> v) {
    const size_t n = v.size(), hi = n / 2;
    std::nth_element(v.begin(), v.begin() + hi, v.end());
    const float b = v[hi];
    if (n & 1) return b;
    const float a = *std::max_element(v.begin(), v.begin() + hi);
    return (a + b) / 2.0f;  // np.mean of the two middle float32 values
}
int b4d_foreground_mask_u16(b4d_handle *, const uint16_t *in, int64_t n, const int64_t shape[3],
                            const float *offsets, float k, int dilate, uint8_t *out, int, int) {
    if (!in || !shape || !offsets || !out || n < 1 || dilate < 0) return fail(B4D_ERR_INVALID, "bad argument");
    const int64_t D = shape[0], H = shape[1], W = shape[2], V = D * H * W;
    std::vector<float> raw((size_t)V), dev((size_t)V);
    std::vector<uint8_t> cur((size_t)V), nxt((size_t)V);
    for (int64_t i = 0; i < n; ++i) {
        for (int64_t v = 0; v < V; ++v) raw[v] = (float)in[i * V + v] - offsets[i];
        const float med = median_f32(raw);
        for (int64_t v = 0; v < V; ++v) dev[v] = std::fabs(raw[v] - med);
        const float mad = median_f32(dev) + 1e-6f;
        const float sigma = 1.4826f * mad;
        const float thr = med + k * sigma;
        for (int64_t v = 0; v < V; ++v) cur[v] = raw[v] > thr;
        for (int it = 0; it < dilate; ++it) {
            for (int64_t z = 0; z < D; ++z)
                for (int64_t y = 0; y < H; ++y)
                    for (int64_t x = 0; x < W; ++x) {
                        const int64_t c = (z * H + y) * W + x;
                        uint8_t m = cur[c];
                        if (z > 0) m |= cur[c - H * W];
                        if (z + 1 < D) m |= cur[c + H * W];
                        if (y > 0) m |= cur[c - W];
                        if (y + 1 < H) m |= cur[c + W];
                        if (x > 0) m |= cur[c - 1];
                        if (x + 1 < W) m |= cur[c + 1];
                        nxt[c] = m;
                    }
            cur.swap(nxt);
        }
        std::memcpy(out + i * V, cur.data(), (size_t)V);
    }
    return 0;
}
int b4d_chunk_shuffle_u16(b4d_handle *, const uint16_t *in, const int64_t shape[3], const int64_t chunk[3],
                          uint8_t *out, uint32_t *hist, int, int) {
    // restatement of the chunk loop of compute_cratio (img_util.py:427-438) + Blosc SHUFFLE, typesize 2
    if (!in || !shape || !chunk || (!out && !hist)) return fail(B4D_ERR_INVALID, "NULL argument");
    const int64_t D = shape[0], H = shape[1], W = shape[2];
    int64_t pos = 0, piece = 0;
    for (int64_t z0 = 0; z0 < D; z0 += chunk[0])
        for (int64_t y0 = 0; y0 < H; y0 += chunk[1])
            for (int64_t x0 = 0; x0 < W; x0 += chunk[2], ++piece) {
                const int64_t dz = std::min(chunk[0], D - z0), dy = std::min(chunk[1], H - y0),
                              dx = std::min(chunk[2], W - x0), ne = dz * dy * dx;
                if (hist) std::memset(hist + piece * 512, 0, 512 * sizeof(uint32_t));
                int64_t e = 0;
                for (int64_t z = 0; z < dz; ++z)
                    for (int64_t y = 0; y < dy; ++y)
                        for (int64_t x = 0; x < dx; ++x, ++e) {
                            const uint16_t v = in[((z0 + z) * H + y0 + y) * W + x0 + x];
                            if (out) {
                                out[pos + e] = (uint8_t)(v & 0xFF);
                                out[pos + ne + e] = (uint8_t)(v >> 8);
                            }
                            if (hist) {
                                ++hist[piece * 512 + (v & 0xFF)];
                                ++hist[piece * 512 + 256 + (v >> 8)];
                            }
                        }
                pos += 2 * ne;
            }
    return 0;
}
int b4d_targets_u16(b4d_handle *hh, const uint16_t *in, int64_t n, const int64_t shape[3], const float *offsets,
                    float sigma, float max_count, float *raw_out, float *teacher_out, int, int) {
    // restatement of data_handling.py:353-354, :332-333 over the oracle's own float32 entry point
    if (!in || !offsets || !teacher_out || n < 1) return fail(B4D_ERR_INVALID, "NULL argument");
    const int64_t V = shape[0] * shape[1] * shape[2];
    std::vector<float> raw((size_t)V);
    for (int64_t i = 0; i < n; ++i) {
        for (int64_t v = 0; v < V; ++v) raw[v] = (float)in[i * V + v] - offsets[i];
        if (raw_out) std::memcpy(raw_out + i * V, raw.data(), (size_t)V * sizeof(float));
        int rc = b4d_denoise_f32(hh, raw.data(), 1, shape, sigma, teacher_out + i * V, 0, 0);
        if (rc) return rc;
        for (int64_t v = 0; v < V; ++v)
            teacher_out[i * V + v] = std::min(std::max(teacher_out[i * V + v], 0.0f), max_count);
    }
    return 0;
}
// the two-call slab form exists for multi-GPU exchange only; the oracle has the one-call form
int b4d_slab_stage1_u16(b4d_handle *, const uint16_t *, const int64_t *, int64_t, int64_t, float, int) {
    return fail(B4D_ERR_UNSUPPORTED, "oracle: use b4d_denoise_slab_u16");
}
int b4d_slab_basic_planes(b4d_handle *, int64_t, int64_t, float *, int, int) {
    return fail(B4D_ERR_UNSUPPORTED, "oracle: use b4d_denoise_slab_u16");
}
int b4d_slab_stage2(b4d_handle *, int64_t, int64_t, float *, int) {
    return fail(B4D_ERR_UNSUPPORTED, "oracle: use b4d_denoise_slab_u16");
}
float *b4d_slab_basic_ptr(b4d_handle *) { return nullptr; }
int b4d_slab_stage2_begin(b4d_handle *, int64_t, int64_t) {
    return fail(B4D_ERR_UNSUPPORTED, "oracle: use b4d_denoise_slab_u16");
}
int b4d_last_timings(b4d_handle *, float *, int64_t *) {
    return fail(B4D_ERR_UNSUPPORTED, "no device timings in the oracle");
}
int b4d_measure_pipe_peaks(b4d_handle *, double *) {
    return fail(B4D_ERR_UNSUPPORTED, "no device in the oracle");
}
// oracle-only: the stage-2 match lists (window index per match [R][K], group size [R]) of the last two-stage
// single-volume call, for the test that traces every large float32-vs-float64 difference to a flipped match
int b4d_oracle_stage2_matches(b4d_handle *hh, uint16_t *widx, uint8_t *cnt, int64_t refs) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || !widx || !cnt || (int64_t)h->last_cnt2.size() != refs)
        return fail(B4D_ERR_INVALID, "no stage-2 match lists of that size");
    std::memcpy(widx, h->last_widx2.data(), h->last_widx2.size() * sizeof(uint16_t));
    std::memcpy(cnt, h->last_cnt2.data(), h->last_cnt2.size());
    return 0;
}
// oracle-only: the matching map denoise_one matches n float32 values with (after the centring of a large DC
// level, which *centre receives), for the tests that assert which map a volume takes
int b4d_oracle_match_map(const float *z, int64_t n, float sigma, int *integral, float *scale, float *centre) {
    if (!z || n < 1 || !integral || !scale || !centre) return fail(B4D_ERR_INVALID, "NULL argument or n < 1");
    MatchMap mm = derive_match_map(z, n, sigma, centre);
    if (*centre != 0.0f) {
        std::vector<float> shifted(n);
        for (int64_t i = 0; i < n; ++i) shifted[i] = z[i] + (-*centre);
        mm = derive_match_map(shifted.data(), n, sigma);
    }
    *integral = mm.integral;
    *scale = mm.scale;
    return 0;
}
int b4d_debug_accumulators(b4d_handle *hh, int64_t *numq, int64_t *wmap, int64_t n) {
    auto *h = reinterpret_cast<b4d_handle_impl *>(hh);
    if (!h || !numq || !wmap || (int64_t)h->last_numq.size() != n)
        return fail(B4D_ERR_INVALID, "no mirror accumulators of that size");
    std::memcpy(numq, h->last_numq.data(), (size_t)n * sizeof(int64_t));
    std::memcpy(wmap, h->last_wmap.data(), (size_t)n * sizeof(int64_t));
    return 0;
}

}  // extern "C"
