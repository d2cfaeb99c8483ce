// b4d_api.cu — the C ABI of include/b4d.h (and b4d_noise.h) over the sm_100a kernels: handle,
// scratch buffers, the two-stage pipeline, slab geometry, statistics.
//
// There is NO CPU fallback here: every entry point that computes needs a CUDA
// device and fails with B4D_ERR_CUDA otherwise.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "b4d_common.cuh"
#include "b4d_host.cuh"

namespace {

thread_local std::string g_err;
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CU_TRY(call)                                                                                  \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess)                                                                        \
            return fail(e_ == cudaErrorMemoryAllocation ? B4D_ERR_NOMEM : B4D_ERR_CUDA,               \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                         \
    } while (0)
#define B4D_TRY(call)        \
    do {                     \
        int rc_ = (call);    \
        if (rc_) return rc_; \
    } while (0)

constexpr int L = 4;
constexpr long long CHUNK_VOXELS = 1342177280ll;  // default: 1.25 Gi voxels per pass (about 45 B of scratch each)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(B4D_ERR_NOMEM, "cudaMalloc(" + std::to_string(bytes) + " B): " + cudaGetErrorString(e));
        }
        cap = bytes;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T *as() const {
        return reinterpret_cast<T *>(p);
    }
};

// u = clamp(int(rint((z + cf) * scale)) + ishift, 0, 65535); see oracle MatchMap.
struct MatchMap {
    float cf = 0.0f, scale = 1.0f;
    int ishift = 0;
    int integral = 1;
};

// Geometry of one pass: `nvol` volumes of D x H x W and the reference-block origins of each stage along z.
struct Plan {
    int D, H, W, nvol;
    std::vector<int> rz1, rz2, ry, rx;
};

// Two-call slab form: what b4d_slab_stage2_begin already launched of the stage-2 front end (planes [o0, o1) of
// the matching image, cell planes [cz0, cz1), tile layers [tz0, tz1) classified and matched).
struct OwnedFront {
    bool done = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // device time of part 1, added to the stage-2 matching slot
    int o0 = 0, o1 = 0, cz0 = 0, cz1 = 0, tz0 = 0, tz1 = 0;
};

}  // namespace

struct b4d_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // host transfers (and the normalise of finished planes) overlapped with kernels
    b4d_profile prof;
    DevBuf coh_x, coh_sm, coh_tmp, coh_keys, coh_sums, coh_lab, coh_w;
    DevBuf in, u16, zf, numq, gmap, basic, out, widx, cnt, ssd, refs, hist, partial, sink, stats, s2, cells, tcls;
    DevBuf alt_in, alt_zf, alt_out, alt_partial, alt_sink;  // second buffer set of b4d_targets_u16
    DevBuf nz_hist, nz_sel, nz_res, nz_full;  // b4d_noise_sigma_u16: per-tile digit histograms, selections, results
    float t_ms[B4D_T_COUNT];
    int64_t launches[B4D_T_COUNT];
    unsigned long long match_stats[4];
    long long pass_voxels = CHUNK_VOXELS;  // voxels per pass (b4d_set_pass_voxels)
    long long pipeline_min_voxels = 1ll << 26;  // host transfers are pipelined from this volume size up
    HostMover mover;  // pageable host arrays <-> device (pinned ring + copy threads)
    // coloured noise (b4d_set_noise_model): relative coefficient variances of both transforms, or white
    bool psd = false;
    float nu_ht[64], nu_wie[64];
    // state between b4d_slab_stage1_u16 and b4d_slab_stage2: the slab (planes from slab_z_begin on) and its map
    bool slab_open = false;
    Plan slab;
    int64_t slab_z_begin = 0;
    float slab_sigma = 0.f;
    MatchMap slab_mm;
    OwnedFront pre;
};

namespace {

// user buffer -> device / device -> user buffer on stream `cs`; host buffers go through the HostMover
cudaError_t copy_in(b4d_handle *h, void *dev, const void *user, size_t bytes, int user_on_device, cudaStream_t cs) {
    if (user_on_device) return cudaMemcpyAsync(dev, user, bytes, cudaMemcpyDeviceToDevice, cs);
    return h->mover.h2d(dev, user, bytes, cs);
}
cudaError_t copy_out(b4d_handle *h, void *user, const void *dev, size_t bytes, int user_on_device, cudaStream_t cs) {
    if (user_on_device) return cudaMemcpyAsync(user, dev, bytes, cudaMemcpyDeviceToDevice, cs);
    return h->mover.d2h(user, dev, bytes, cs);
}

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
    if (p.block != 4 || p.step != 3) return fail(B4D_ERR_UNSUPPORTED, "only block = 4, step = 3 are implemented");
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
int check_shape(const int64_t shape[3]) {
    for (int i = 0; i < 3; ++i)
        if (shape[i] < L || shape[i] > 65535) return fail(B4D_ERR_INVALID, "every dimension must be in [4, 65535]");
    return 0;
}

// Reference-block origins along one axis: 0, 3, 6, ... plus N-4 (SURVEY App. A).
std::vector<int> ref_origins(int64_t n) {
    std::vector<int> o;
    for (int64_t v = 0; v + L <= n; v += 3) o.push_back((int)v);
    if ((n - L) % 3 != 0) o.push_back((int)(n - L));
    return o;
}
std::vector<int> slab_origins(int64_t z_total, int64_t z_begin, int64_t depth, int r) {
    std::vector<int> o;
    for (int gz : ref_origins(z_total)) {
        const int64_t lo = std::max<int64_t>(0, gz - r);
        const int64_t hi = std::min<int64_t>(z_total - L, gz + r) + (L - 1);
        if (lo >= z_begin && hi < z_begin + depth) o.push_back((int)(gz - z_begin));
    }
    return o;
}

double bessel_i0(double x) {
    double s = 1.0, t = 1.0;
    for (int k = 1; k < 64; ++k) {
        t *= (x / (2.0 * k)) * (x / (2.0 * k));
        s += t;
        if (t < 1e-18 * s) break;
    }
    return s;
}
B4dTables make_tables(const b4d_profile &p, float sigma, const float *nu_ht = nullptr, const float *nu_wie = nullptr) {
    B4dTables t;
    std::memset(&t, 0, sizeof(t));
    // coloured-noise tables (white: nu = 1): identical code in oracle/b4d_oracle.cpp make_tables
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
    float kf[4];
    for (int n = 0; n < 4; ++n) {
        double w = 1.0;
        if (p.kaiser_beta > 0) {
            const double a = 2.0 * n / 3.0 - 1.0;
            w = bessel_i0((double)p.kaiser_beta * std::sqrt(std::max(0.0, 1.0 - a * a))) /
                bessel_i0((double)p.kaiser_beta);
        }
        kf[n] = (float)w;
        t.kf[n] = kf[n];
    }
    for (int z = 0; z < 4; ++z)
        for (int y = 0; y < 4; ++y)
            for (int x = 0; x < 4; ++x) {
                volatile float zy = kf[z] * kf[y];  // two separately rounded float32 products
                volatile float zyx = zy * kf[x];
                t.win[(z * 4 + y) * 4 + x] = zyx;
            }
    for (int m = 0; m < 16; ++m) {
        const double s = std::ldexp(1.0, m / 2) * ((m & 1) ? M_SQRT2 : 1.0);
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
    volatile float s2 = sigma * sigma;
    t.sigma2 = s2;
    return t;
}

int centre_shift(double lo, double hi) { return (int)(std::floor((65535.0 - (hi - lo)) * 0.5) - lo); }

int tau_for(float tau, float sigma, float scale, int Ns, uint32_t *out) {
    const double s = (double)sigma * (double)scale;
    const double v = std::floor((double)tau * s * s * 64.0);
    const int kb = (Ns * Ns * Ns <= 2048) ? 11 : 12;
    const double lim = std::ldexp(1.0, 32 - kb) - 2.0;
    if (!(v <= lim))
        return fail(B4D_ERR_UNSUPPORTED,
                    "tau*sigma^2*64 = " + std::to_string(v) + " exceeds the 32-bit match key (" +
                        std::to_string(lim) + "); lower sigma or tau");
    *out = (uint32_t)v;
    return 0;
}

// Planes [z_begin, z_begin + shape[0]) of a z_total-plane volume: the reference origins along z of each stage are
// those of the whole volume whose search window lies inside the slab (a whole volume: z_begin = 0, z_total = D).
Plan make_plan(const int64_t shape[3], int64_t z_begin, int64_t z_total, int nvol, const b4d_profile &p) {
    Plan pl;
    pl.D = (int)shape[0];
    pl.H = (int)shape[1];
    pl.W = (int)shape[2];
    pl.nvol = nvol;
    pl.rz1 = slab_origins(z_total, z_begin, shape[0], p.search_ht / 2);
    pl.rz2 = slab_origins(z_total, z_begin, shape[0], p.search_wie / 2);
    pl.ry = ref_origins(shape[1]);
    pl.rx = ref_origins(shape[2]);
    return pl;
}

void fill_geom(const Plan &pl, const std::vector<int> &rz, const int *d_refs, B4dGeom *g) {
    g->D = pl.D;
    g->H = pl.H;
    g->W = pl.W;
    g->nvol = pl.nvol;
    g->nrz = (int)rz.size();
    g->nry = (int)pl.ry.size();
    g->nrx = (int)pl.rx.size();
    g->tz = (g->nrz + 3) / 4;
    g->ty = (g->nry + 3) / 4;
    g->tx = (g->nrx + 3) / 4;
    g->refz = d_refs;
    g->refy = d_refs + rz.size();
    g->refx = d_refs + rz.size() + pl.ry.size();
    g->vol_stride = (long long)pl.D * pl.H * pl.W;
    g->refs_per_vol = (long long)g->nrz * g->nry * g->nrx;
}

// The reference-origin lists of both stages on the device, [rz1 | ry | rx | rz2 | ry | rx], and their geometry.
int upload_geometry(b4d_handle *h, const Plan &pl, B4dGeom *g1, B4dGeom *g2) {
    std::vector<int> refs;
    refs.insert(refs.end(), pl.rz1.begin(), pl.rz1.end());
    refs.insert(refs.end(), pl.ry.begin(), pl.ry.end());
    refs.insert(refs.end(), pl.rx.begin(), pl.rx.end());
    const size_t off2 = refs.size();
    refs.insert(refs.end(), pl.rz2.begin(), pl.rz2.end());
    refs.insert(refs.end(), pl.ry.begin(), pl.ry.end());
    refs.insert(refs.end(), pl.rx.begin(), pl.rx.end());
    B4D_TRY(h->refs.ensure(refs.size() * sizeof(int)));
    CU_TRY(cudaMemcpyAsync(h->refs.p, refs.data(), refs.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU_TRY(cudaStreamSynchronize(h->stream));  // `refs` is a stack vector
    fill_geom(pl, pl.rz1, h->refs.as<int>(), g1);
    fill_geom(pl, pl.rz2, h->refs.as<int>() + off2, g2);
    const long long R1 = g1->refs_per_vol * pl.nvol, R2 = g2->refs_per_vol * pl.nvol;
    if ((long long)pl.nvol * g1->tz * g1->ty * g1->tx > 2147483647ll || (R1 + 3) / 4 > 2147483647ll ||
        (R2 + 3) / 4 > 2147483647ll)
        return fail(B4D_ERR_TOO_LARGE, "too many reference blocks for one launch");
    return 0;
}

// Ordering events owned for the duration of one call: destroyed on every exit path.
struct EventSet {
    std::vector<cudaEvent_t> evs;
    EventSet() = default;
    EventSet(const EventSet &) = delete;
    EventSet &operator=(const EventSet &) = delete;
    ~EventSet() {
        for (auto e : evs) cudaEventDestroy(e);
    }
    cudaError_t make(cudaEvent_t *out) {
        const cudaError_t e = cudaEventCreateWithFlags(out, cudaEventDisableTiming);
        if (e == cudaSuccess) evs.push_back(*out);
        return e;
    }
};

// One stage boundary timing: we record an event after each kernel family and
// resolve all of them after the final synchronise.
struct StageClock {
    b4d_handle *h;
    std::vector<cudaEvent_t> evs;
    std::vector<std::pair<int, int>> tags;  // (slot, launches) for interval i -> i+1
    explicit StageClock(b4d_handle *hh) : h(hh) {}
    StageClock(const StageClock &) = delete;
    StageClock &operator=(const StageClock &) = delete;
    ~StageClock() {  // an error return before resolve()
        for (auto e : evs) cudaEventDestroy(e);
    }
    void mark(int slot, int launches) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, h->stream);
        evs.push_back(e);
        tags.push_back({slot, launches});
    }
    void resolve() {
        for (size_t i = 1; i < evs.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, evs[i - 1], evs[i]);
            const int slot = tags[i].first;
            if (slot >= 0 && slot < B4D_T_COUNT) {
                h->t_ms[slot] += ms;
                h->launches[slot] += tags[i].second;
            }
        }
        for (auto e : evs) cudaEventDestroy(e);
        evs.clear();
        tags.clear();
    }
};

// Where the result goes when it is wanted in HOST memory: planes [p0, p1) of the (single) volume, to `host`
// (p1 - p0 planes).  stage2_back then runs the filter in z chunks and every chunk of finished planes is
// normalised and copied out on a second stream while the next chunks still compute — the device-to-host copy
// (4 B/voxel over PCIe) hides behind the filter.
struct HostSink {
    void *host = nullptr;  // float32, or uint16 with a QuantSpec
    long long p0 = 0, p1 = 0;
    bool done = false;  // set when stage2_back delivered the result itself
};
// Fused K6 + K7: the last normalise writes q = quantize(result) as uint16 instead of the float32 result
// (the pass's `out` then points at uint16 storage; 2 B/voxel leave the device instead of 4).
struct QuantSpec {
    float sub = 0.f, add = 0.f, step = 1.f;
    int trunc = 0;
};

constexpr int UPLOAD_CHUNKS = 8;
// Chunked launches under-fill the GPU on small volumes (a 128^3 patch ran 1.5x slower in 8 chunks and its
// whole upload takes 0.1 ms), so the transfers are pipelined only from `pipeline_min_voxels` up.
bool can_stream_upload(const b4d_handle *h, const Plan &pl) {
    return pl.nvol == 1 && ((long long)pl.H * pl.W) % 8 == 0 && pl.D >= 16 * UPLOAD_CHUNKS &&
           (long long)pl.D * pl.H * pl.W >= h->pipeline_min_voxels && !pl.rz1.empty();
}

// The two-word min / max sink of the uint16 conversion kernels: reset before the launch, read back after it
// (this synchronises `s`).
int range_reset(DevBuf &sink, cudaStream_t s) {
    B4D_TRY(sink.ensure(64));
    const unsigned init[2] = {0xFFFFu, 0u};
    CU_TRY(cudaMemcpyAsync(sink.p, init, sizeof(init), cudaMemcpyHostToDevice, s));
    return 0;
}
int range_read(const DevBuf &sink, cudaStream_t s, double *lo, double *hi) {
    unsigned got[2] = {0, 0};
    CU_TRY(cudaMemcpyAsync(got, sink.p, sizeof(got), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    *lo = got[0];
    *hi = got[1];
    return 0;
}

// One pass of the two-stage pipeline over device-resident volumes, set up once per call by make_pass:
//   zf     float32 noisy volumes            [nvol*V]
//   u      uint16 matching image of stage 1 [nvol*V]   (overwritten by that of stage 2)
//   basic  float32 basic estimate           [nvol*V]   (h->basic, or `out` when profile.stages = 1)
//   out    result                           [nvol*V]   (float32, or uint16 with a QuantSpec)
struct Pass {
    b4d_handle *h;
    const Plan *pl;
    StageClock *clk;
    MatchMap mm;  // a streamed stage-1 upload sets ishift from the data range
    float *zf;
    uint16_t *u;
    float *basic, *out;
    long long TV, R1, R2;  // voxels and reference blocks of each stage, all volumes
    B4dGeom g1, g2;
    B4dTables tab;
    MatchParams mp1, mp2;
    FilterParams fp1, fp2;
};

int make_pass(b4d_handle *h, const Plan &pl, float sigma, const MatchMap &mm, float *zf, uint16_t *u, float *out,
              StageClock &clk, Pass &ps) {
    const b4d_profile &p = h->prof;
    uint32_t tau1 = 0, tau2 = 0;
    B4D_TRY(tau_for(p.tau_ht, sigma, mm.scale, p.search_ht, &tau1));
    if (p.stages == 2) B4D_TRY(tau_for(p.tau_wie, sigma, mm.scale, p.search_wie, &tau2));
    B4D_TRY(upload_geometry(h, pl, &ps.g1, &ps.g2));
    ps.h = h;
    ps.pl = &pl;
    ps.clk = &clk;
    ps.mm = mm;
    ps.zf = zf;
    ps.u = u;
    ps.out = out;
    ps.TV = (long long)pl.D * pl.H * pl.W * pl.nvol;
    ps.R1 = ps.g1.refs_per_vol * pl.nvol;
    ps.R2 = ps.g2.refs_per_vol * pl.nvol;
    const long long Rmax = std::max(ps.R1, ps.R2);
    B4D_TRY(h->widx.ensure((size_t)Rmax * std::max(p.k_ht, p.k_wie) * sizeof(uint16_t)));
    B4D_TRY(h->cnt.ensure((size_t)Rmax));
    B4D_TRY(h->basic.ensure((size_t)ps.TV * sizeof(float)));
    B4D_TRY(h->s2.ensure((size_t)ps.TV * sizeof(uint2)));
    const size_t ncell = (size_t)pl.nvol * pl.D * ps.g1.ty * ps.g1.tx;  // per-plane window ranges of every tile
    const size_t ntile = (size_t)pl.nvol * std::max(ps.g1.tz, ps.g2.tz) * ps.g1.ty * ps.g1.tx;
    B4D_TRY(h->cells.ensure(ncell * sizeof(uint32_t)));
    B4D_TRY(h->tcls.ensure(ntile * sizeof(uint32_t)));
    B4D_TRY(h->stats.ensure(4 * sizeof(unsigned long long)));
    // Both stages aggregate in order-independent fixed point (int64): the result does not
    // depend on scheduling, a slab equals the whole volume bit for bit, and the basic estimate
    // that feeds the stage-2 matching (a discontinuous decision) is reproducible.
    // profile.deterministic is kept in the ABI and is always honoured.
    B4D_TRY(h->numq.ensure((size_t)ps.TV * sizeof(long long)));
    B4D_TRY(h->gmap.ensure((size_t)ps.TV * sizeof(uint32_t)));
    ps.tab = make_tables(p, sigma, h->psd ? h->nu_ht : nullptr, h->psd ? h->nu_wie : nullptr);
    if (h->psd && (p.search_ht > 11 || p.search_wie > 11))
        return fail(B4D_ERR_UNSUPPORTED, "a coloured-noise model needs search windows of at most 11");
    b4d_upload_tables(ps.tab, h->stream);  // on every call: the tables are shared by all handles
    ps.basic = p.stages == 1 ? out : h->basic.as<float>();

    MatchParams &mp = ps.mp1;
    mp.g = ps.g1;
    mp.u = u;
    mp.s21 = h->s2.as<uint2>();
    mp.cells = h->cells.as<uint32_t>();
    mp.tcls = h->tcls.as<uint32_t>();
    mp.tau = tau1;
    mp.K = p.k_ht;
    mp.widx = h->widx.as<uint16_t>();
    mp.cnt = h->cnt.as<uint8_t>();
    mp.ssd_out = nullptr;
    mp.stats = h->stats.as<unsigned long long>();
    ps.mp2 = mp;
    ps.mp2.g = ps.g2;
    ps.mp2.tau = tau2;
    ps.mp2.K = p.k_wie;

    FilterParams &fp = ps.fp1;
    fp.g = ps.g1;
    fp.zf = zf;
    fp.basic = nullptr;
    fp.widx = mp.widx;
    fp.cnt = mp.cnt;
    fp.K = p.k_ht;
    fp.Ns = p.search_ht;
    fp.nseg = 1;
    fp.psd = h->psd ? 1 : 0;
    fp.qscale = mm.scale;  // data * scale spans at most the 16-bit matching range: terms stay below 2^39
    fp.numq = h->numq.as<long long>();
    fp.gmap = h->gmap.as<uint32_t>();
    ps.fp2 = fp;
    ps.fp2.g = ps.g2;
    ps.fp2.basic = ps.basic;
    ps.fp2.K = p.k_wie;
    ps.fp2.Ns = p.search_wie;
    return 0;
}

int zero_acc(const Pass &ps) {
    CU_TRY(cudaMemsetAsync(ps.h->numq.p, 0, (size_t)ps.TV * sizeof(long long), ps.h->stream));
    CU_TRY(cudaMemsetAsync(ps.h->gmap.p, 0, (size_t)ps.TV * sizeof(uint32_t), ps.h->stream));
    return 0;
}

// Planes [z0, z1) of every volume of the accumulators divided out: num / den from `fallback` into `dst`, or
// quantized into `dst` as uint16 with `q`.
void normalise(const Pass &ps, const float *fallback, float *dst, int z0, int z1, const QuantSpec *q, cudaStream_t s) {
    const Plan &pl = *ps.pl;
    const long long *numq = ps.h->numq.as<long long>();
    const uint32_t *gmap = ps.h->gmap.as<uint32_t>();
    if (q)
        b4d_launch_normalise_q16(numq, gmap, fallback, reinterpret_cast<uint16_t *>(dst), pl.D, pl.H, pl.W, pl.nvol,
                                 z0, z1, 1.0f / ps.mm.scale, ps.tab.kf, q->sub, q->add, q->step, q->trunc, s);
    else
        b4d_launch_normalise_wm(numq, gmap, fallback, dst, pl.D, pl.H, pl.W, pl.nvol, z0, z1, 1.0f / ps.mm.scale,
                                ps.tab.kf, s);
}

// Stage-1 front end of one uint16 volume in host memory: it is uploaded in z chunks on the copy stream and the
// float conversion, block energies, tile classification and matching follow chunk by chunk, so that the
// host-to-device copy (2 B/voxel over PCIe) hides behind the stage-1 matcher.  The data range sets the centre
// shift of the stage-2 matching image.
int stage1_streamed_front(Pass &ps, const uint16_t *host_src) {
    b4d_handle *h = ps.h;
    const Plan &pl = *ps.pl;
    const b4d_profile &p = h->prof;
    cudaStream_t s = h->stream;
    const long long P = (long long)pl.H * pl.W;
    const int E = p.search_ht + 12, cd = (pl.D + 3) / 4;
    B4D_TRY(range_reset(h->sink, s));
    EventSet owned;
    cudaEvent_t evs[UPLOAD_CHUNKS];
    int zprev = 0, odone = 0, cdone = 0, tdone = 0;
    for (int k = 0; k < UPLOAD_CHUNKS; ++k) {
        int zu = (k + 1 == UPLOAD_CHUNKS) ? pl.D : (int)(((long long)(k + 1) * pl.D / UPLOAD_CHUNKS + 3) & ~3ll);
        zu = std::min(zu, pl.D);
        CU_TRY(copy_in(h, ps.u + zprev * P, host_src + zprev * P, (size_t)(zu - zprev) * P * sizeof(uint16_t), 0,
                       h->copy_stream));
        CU_TRY(owned.make(&evs[k]));
        CU_TRY(cudaEventRecord(evs[k], h->copy_stream));
        CU_TRY(cudaStreamWaitEvent(s, evs[k], 0));
        // planes [0, zu) are on the device: everything that needs no plane beyond zu - 1
        b4d_launch_u16_to_f32(ps.u + zprev * P, ps.zf + zprev * P, (long long)(zu - zprev) * P, h->sink.as<unsigned>(),
                              s);
        const int o1 = (zu == pl.D) ? pl.D - 3 : zu - 3;            // block origins with all 4 planes present
        b4d_launch_block_energy_range(ps.u, h->s2.as<uint2>(), pl.D, pl.H, pl.W, 1, odone, o1, s);
        odone = std::max(odone, o1);
        const int c1 = (zu == pl.D) ? cd : zu / 4;                   // complete 4-plane cells
        int t1 = tdone;                                              // tile layers whose neighbourhood is complete
        while (t1 < ps.g1.tz && std::min(pl.rz1[4 * t1] - p.search_ht / 2 + E - 1, pl.D - 1) < zu) ++t1;
        b4d_launch_match_range(ps.mp1, p.search_ht, cdone, c1, (long long)tdone * ps.g1.ty * ps.g1.tx,
                               (long long)t1 * ps.g1.ty * ps.g1.tx, s);
        cdone = c1;
        tdone = t1;
        zprev = zu;
    }
    double lo = 0, hi = 0;
    B4D_TRY(range_read(h->sink, s, &lo, &hi));
    ps.mm.ishift = centre_shift(lo, hi);
    return 0;
}

// Stage 1, hard thresholding: block energies and matching on the uint16 image, filter, normalise into the basic
// estimate.  `host_src`: the uint16 volume is still in host memory and is uploaded here (can_stream_upload
// holds).  `fuse_match`: the normalise also writes the stage-2 matching image rint(basic * scale) + shift, so that
// the separate conversion pass (4 B read + 2 B write per voxel) is not needed.
int stage1(Pass &ps, const uint16_t *host_src, bool fuse_match) {
    b4d_handle *h = ps.h;
    const Plan &pl = *ps.pl;
    const b4d_profile &p = h->prof;
    cudaStream_t s = h->stream;
    StageClock &clk = *ps.clk;
    CU_TRY(cudaMemsetAsync(h->stats.p, 0, 4 * sizeof(unsigned long long), s));
    B4D_TRY(zero_acc(ps));
    clk.mark(B4D_T_PREP, 1);
    if (!host_src) b4d_launch_block_energy(ps.u, h->s2.as<uint2>(), pl.D, pl.H, pl.W, pl.nvol, s);
    clk.mark(B4D_T_K0, 1);
    if (host_src)
        B4D_TRY(stage1_streamed_front(ps, host_src));
    else if (ps.R1 > 0)
        b4d_launch_match(ps.mp1, p.search_ht, s);
    clk.mark(B4D_T_MATCH1, 4);
    if (ps.R1 > 0) b4d_launch_filter(ps.fp1, false, s);
    clk.mark(B4D_T_FILTER1, 1);
    if (fuse_match)
        b4d_launch_normalise_match(h->numq.as<long long>(), h->gmap.as<uint32_t>(), ps.zf, ps.basic, ps.u,
                                   ps.mm.scale, ps.mm.ishift, pl.D, pl.H, pl.W, pl.nvol, 1.0f / ps.mm.scale,
                                   ps.tab.kf, s);
    else
        normalise(ps, ps.zf, ps.basic, 0, pl.D, nullptr, s);
    clk.mark(B4D_T_NORM1, 1);
    CU_TRY(cudaGetLastError());
    return 0;
}

// Stage-2 front end on the whole basic estimate: its matching image (unless stage 1 already wrote it), block
// energies, matching.
int stage2_front_whole(Pass &ps, bool already_converted) {
    b4d_handle *h = ps.h;
    const Plan &pl = *ps.pl;
    cudaStream_t s = h->stream;
    if (!already_converted) b4d_launch_to_match(ps.basic, ps.u, ps.TV, 0.0f, ps.mm.scale, ps.mm.ishift, s);
    B4D_TRY(zero_acc(ps));
    ps.clk->mark(B4D_T_PREP, 2);
    b4d_launch_block_energy(ps.u, h->s2.as<uint2>(), pl.D, pl.H, pl.W, pl.nvol, s);
    ps.clk->mark(B4D_T_K0, 1);
    if (ps.R2 > 0) b4d_launch_match(ps.mp2, h->prof.search_wie, s);
    ps.clk->mark(B4D_T_MATCH2, 4);
    return 0;
}

// Two-call slab form, part 1 (b4d_slab_stage2_begin): everything of the stage-2 front end that reads no plane
// outside the owned planes [o0, o1) — the planes a neighbour exchange is about to overwrite lie outside.
// Launched and left running: the exchange overlaps it.  h->pre records the ranges for stage2_front_rest.
int stage2_front_owned(Pass &ps, int o0, int o1) {
    b4d_handle *h = ps.h;
    const Plan &pl = *ps.pl;
    cudaStream_t s = h->stream;
    OwnedFront &f = h->pre;
    const long long Pv = (long long)pl.H * pl.W, tiles_per_layer = (long long)ps.g2.ty * ps.g2.tx;
    const int E2 = h->prof.search_wie + 12, r2 = h->prof.search_wie / 2;
    f.o0 = o0;
    f.o1 = o1;
    f.cz0 = (o0 + 3) / 4;
    f.cz1 = (o1 == pl.D) ? (pl.D + 3) / 4 : o1 / 4;
    auto layer_inside = [&](int tz) {
        const int bz = pl.rz2[4 * tz] - r2;
        const int zlo = std::max(bz, 0), zhi = std::min(bz + E2 - 1, pl.D - 1);
        return zlo / 4 >= f.cz0 && zhi / 4 < f.cz1 && zlo >= o0 && zhi < o1;
    };
    f.tz0 = 0;
    while (f.tz0 < ps.g2.tz && !layer_inside(f.tz0)) ++f.tz0;
    f.tz1 = f.tz0;
    while (f.tz1 < ps.g2.tz && layer_inside(f.tz1)) ++f.tz1;
    if (o1 > o0)
        b4d_launch_to_match(ps.basic + o0 * Pv, ps.u + o0 * Pv, (long long)(o1 - o0) * Pv, 0.0f, ps.mm.scale,
                            ps.mm.ishift, s);
    B4D_TRY(zero_acc(ps));
    b4d_launch_block_energy_range(ps.u, h->s2.as<uint2>(), pl.D, pl.H, pl.W, 1, o0, std::max(o0, o1 - 3), s);
    if (ps.R2 > 0)
        b4d_launch_match_range(ps.mp2, h->prof.search_wie, f.cz0, std::max(f.cz0, f.cz1), f.tz0 * tiles_per_layer,
                               f.tz1 * tiles_per_layer, s);
    f.done = true;
    CU_TRY(cudaGetLastError());
    return 0;
}

// Part 2: the rest of the stage-2 front end (planes, origins, cells and tile layers outside the ranges of part 1).
int stage2_front_rest(Pass &ps) {
    b4d_handle *h = ps.h;
    const Plan &pl = *ps.pl;
    cudaStream_t s = h->stream;
    OwnedFront &f = h->pre;
    const long long Pv = (long long)pl.H * pl.W, tiles_per_layer = (long long)ps.g2.ty * ps.g2.tx;
    const int o0 = f.o0, o1 = f.o1;
    if (o0 > 0) b4d_launch_to_match(ps.basic, ps.u, o0 * Pv, 0.0f, ps.mm.scale, ps.mm.ishift, s);
    if (o1 < pl.D)
        b4d_launch_to_match(ps.basic + o1 * Pv, ps.u + o1 * Pv, (pl.D - o1) * Pv, 0.0f, ps.mm.scale, ps.mm.ishift, s);
    b4d_launch_block_energy_range(ps.u, h->s2.as<uint2>(), pl.D, pl.H, pl.W, 1, 0, std::min(o0, pl.D - 3), s);
    b4d_launch_block_energy_range(ps.u, h->s2.as<uint2>(), pl.D, pl.H, pl.W, 1, std::max(o0, o1 - 3), pl.D - 3, s);
    ps.clk->mark(B4D_T_PREP, 4);
    if (ps.R2 > 0) {
        b4d_launch_match_range(ps.mp2, h->prof.search_wie, 0, f.cz0, 0, f.tz0 * tiles_per_layer, s);
        b4d_launch_match_range(ps.mp2, h->prof.search_wie, std::max(f.cz0, f.cz1), (pl.D + 3) / 4,
                               f.tz1 * tiles_per_layer, (long long)ps.g2.tz * tiles_per_layer, s);
    }
    ps.clk->mark(B4D_T_MATCH2, 8);
    f.done = false;
    return 0;
}

// Stage 2, Wiener: the filter and the normalise into `out` (quantized with `q`).  A large single volume whose
// result goes to host memory (`sink`) is filtered in z chunks, see HostSink.
int stage2_back(Pass &ps, HostSink *sink, const QuantSpec *q) {
    b4d_handle *h = ps.h;
    const Plan &pl = *ps.pl;
    cudaStream_t s = h->stream;
    StageClock &clk = *ps.clk;
    const long long P = (long long)pl.H * pl.W;
    constexpr int NCH = 8;
    const int nseg_ch = (sink && sink->host && pl.nvol == 1 && ps.R2 > 0 && (P & 3) == 0 &&
                         ps.TV >= h->pipeline_min_voxels)
                            ? b4d_filter_segments(ps.fp2, true, NCH)
                            : 0;
    if (nseg_ch >= NCH && nseg_ch % NCH == 0) {
        // chunked: launch everything on the compute stream first (events between the chunks), then
        // queue normalise + copy of the planes each chunk finishes on the copy stream
        const int spc = nseg_ch / NCH, r2 = h->prof.search_wie / 2;
        EventSet owned;
        cudaEvent_t evs[NCH];
        for (int c = 0; c < NCH; ++c) {
            b4d_launch_filter_segments(ps.fp2, true, nseg_ch, c * spc, spc, s);
            CU_TRY(owned.make(&evs[c]));
            CU_TRY(cudaEventRecord(evs[c], s));
        }
        clk.mark(B4D_T_FILTER2, NCH);
        const size_t esz = q ? sizeof(uint16_t) : sizeof(float);
        long long zdone = 0;
        for (int c = 0; c < NCH; ++c) {
            // after chunk c: no later segment touches a plane below the window of its first reference
            long long zfin = pl.D;
            if (c + 1 < NCH) {
                const int iz_next = (int)((long long)(c + 1) * spc * ps.g2.nrz / nseg_ch);
                zfin = std::max<long long>(0, (long long)pl.rz2[iz_next] - r2);
            }
            CU_TRY(cudaStreamWaitEvent(h->copy_stream, evs[c], 0));
            if (zfin > zdone) {
                // origins below zfin are final as well: a block touches its own origin plane
                normalise(ps, ps.basic, ps.out, (int)zdone, (int)zfin, q, h->copy_stream);
                const long long a = std::max(zdone, sink->p0), b = std::min(zfin, sink->p1);
                if (b > a)
                    CU_TRY(copy_out(h, static_cast<char *>(sink->host) + (size_t)(a - sink->p0) * P * esz,
                                    reinterpret_cast<char *>(ps.out) + (size_t)a * P * esz, (size_t)(b - a) * P * esz,
                                    0, h->copy_stream));
                zdone = zfin;
            }
        }
        CU_TRY(cudaStreamSynchronize(h->copy_stream));
        clk.mark(B4D_T_NORM2, NCH);
        sink->done = true;
        CU_TRY(cudaGetLastError());
        return 0;
    }
    if (ps.R2 > 0) b4d_launch_filter(ps.fp2, true, s);
    clk.mark(B4D_T_FILTER2, 1);
    normalise(ps, ps.basic, ps.out, 0, pl.D, q, s);
    clk.mark(B4D_T_NORM2, 1);
    CU_TRY(cudaGetLastError());
    return 0;
}

// Both stages of one pass (stage 1 alone when profile.stages = 1).
int denoise_pass(Pass &ps, const uint16_t *host_src, HostSink *sink, const QuantSpec *q) {
    const bool two = ps.h->prof.stages == 2;
    B4D_TRY(stage1(ps, host_src, two));
    if (!two) return 0;
    B4D_TRY(stage2_front_whole(ps, true));
    return stage2_back(ps, sink, q);
}

// float32 input -> matching map (shift, scale); mirrors oracle derive_match_map.
// Float data whose magnitude (in matching steps) is far above its range — a large DC level — would push the
// fixed-point numerator terms (20-bit weight x value) past their 2^39 clamp.  Such inputs are denoised on
// z - c0 and c0 is added back at the end (BM4D is translation equivariant); *centre receives c0, or 0 when no
// centring is needed: count-scale data (|z| <= 65535 at scale 1) never is, so the common paths are untouched.
constexpr double CENTRE_LIMIT = 131072.0;  // 2^17 matching steps
int derive_match_map(b4d_handle *h, const float *d_in, long long n, float sigma, MatchMap *mm, float *centre = nullptr) {
    cudaStream_t s = h->stream;
    float z0 = 0.f;
    CU_TRY(cudaMemcpyAsync(&z0, d_in, sizeof(float), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    const double c = std::rint((double)z0) - (double)z0;
    const int nb = b4d_analyze_blocks();
    B4D_TRY(h->partial.ensure((size_t)nb * 6 * sizeof(double)));
    b4d_launch_analyze(d_in, n, c, h->partial.as<double>(), s);
    std::vector<double> part((size_t)nb * 6);
    CU_TRY(cudaMemcpyAsync(part.data(), h->partial.p, part.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    double dev = 0, lo = 1e300, hi = -1e300, zlo = 1e300, zhi = -1e300, nonfinite = 0;
    for (int b = 0; b < nb; ++b) {
        dev = std::max(dev, part[b * 6 + 0]);
        lo = std::min(lo, part[b * 6 + 1]);
        hi = std::max(hi, part[b * 6 + 2]);
        zlo = std::min(zlo, part[b * 6 + 3]);
        zhi = std::max(zhi, part[b * 6 + 4]);
        nonfinite = std::max(nonfinite, part[b * 6 + 5]);
    }
    if (nonfinite > 0 || !(std::isfinite(zlo) && std::isfinite(zhi)))
        return fail(B4D_ERR_INVALID, "input contains non-finite values (NaN or infinity)");
    if (dev <= 1.0 / 64.0 && hi - lo <= 65535.0) {
        mm->integral = 1;
        mm->scale = 1.0f;
        mm->cf = (float)c;
        mm->ishift = centre_shift(lo, hi);
    } else {
        const double range = std::max(zhi - zlo, 1e-30);
        const int e_range = (int)std::floor(std::log2(65535.0 / range));
        const int e_sigma = (int)std::floor(std::log2(64.0 / (double)sigma));
        mm->integral = 0;
        mm->scale = (float)std::ldexp(1.0, std::min(e_range, e_sigma));
        mm->cf = 0.0f;
        mm->ishift = centre_shift(std::floor(zlo * (double)mm->scale), std::ceil(zhi * (double)mm->scale));
    }
    if (centre) {
        const double peak = std::max(std::fabs(zlo), std::fabs(zhi)) * (double)mm->scale;
        *centre = 0.0f;
        if (peak > CENTRE_LIMIT) *centre = mm->integral ? (float)std::rint(0.5 * (lo + hi)) : (float)(0.5 * (zlo + zhi));
    }
    return 0;
}

// uint16 input: float copy + the centring shift of the stage-2 matching image
// (stage 1 matches on the raw integers; mirrors oracle denoise_one).
int convert_u16(b4d_handle *h, const uint16_t *d_in, float *d_zf, long long n, MatchMap *mm) {
    B4D_TRY(range_reset(h->sink, h->stream));
    b4d_launch_u16_to_f32(d_in, d_zf, n, h->sink.as<unsigned>(), h->stream);
    double lo = 0, hi = 0;
    B4D_TRY(range_read(h->sink, h->stream, &lo, &hi));
    *mm = MatchMap();  // integral, unit scale
    mm->ishift = centre_shift(lo, hi);
    return 0;
}

int common_checks(b4d_handle *h, const void *in, const void *out, const int64_t shape[3], float sigma) {
    if (!h || !in || !out || !shape) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!(sigma > 0) || !std::isfinite(sigma)) return fail(B4D_ERR_INVALID, "sigma must be positive and finite");
    B4D_TRY(check_shape(shape));
    CU_TRY(cudaSetDevice(h->device));
    return 0;
}

void reset_timings(b4d_handle *h) {
    for (int i = 0; i < B4D_T_COUNT; ++i) {
        h->t_ms[i] = 0.f;
        h->launches[i] = 0;
    }
}

// The end of a denoise call: wait for the compute stream, book the stage timings, fetch the matcher statistics.
int finish(b4d_handle *h, StageClock &clk) {
    CU_TRY(cudaStreamSynchronize(h->stream));
    clk.resolve();
    CU_TRY(cudaMemcpy(h->match_stats, h->stats.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return 0;
}

// One uint16 volume or slab in: from host memory and large enough, it stays there for stage 1 to upload behind
// the matcher (*host_src = in); otherwise it is copied to h->in and converted into h->zf with its matching map.
int stage_u16_input(b4d_handle *h, const Plan &pl, const uint16_t *in, int in_on_device, StageClock &clk,
                    MatchMap *mm, const uint16_t **host_src) {
    const long long V = (long long)pl.D * pl.H * pl.W;
    B4D_TRY(h->in.ensure((size_t)V * sizeof(uint16_t)));
    B4D_TRY(h->u16.ensure((size_t)V * sizeof(uint16_t) + 16));
    B4D_TRY(h->zf.ensure((size_t)V * sizeof(float)));
    B4D_TRY(h->out.ensure((size_t)V * sizeof(float)));
    *host_src = nullptr;
    if (!in_on_device && can_stream_upload(h, pl)) {
        *host_src = in;
        clk.mark(-1, 0);
    } else {
        CU_TRY(copy_in(h, h->in.p, in, (size_t)V * sizeof(uint16_t), in_on_device, h->stream));
        clk.mark(-1, 0);
        B4D_TRY(convert_u16(h, h->in.as<uint16_t>(), h->zf.as<float>(), V, mm));
    }
    clk.mark(B4D_T_PREP, 1);
    return 0;
}

// Batched denoise, chunked so scratch stays bounded.
template <class T>
int denoise_batch(b4d_handle *h, const T *in, int64_t n, const int64_t shape[3], float sigma, float *out,
                  int in_dev, int out_dev) {
    B4D_TRY(common_checks(h, in, out, shape, sigma));
    if (n < 1) return fail(B4D_ERR_INVALID, "n must be >= 1");
    reset_timings(h);
    const long long V = shape[0] * shape[1] * shape[2];
    const int64_t per = std::max<int64_t>(1, std::min<int64_t>(n, h->pass_voxels / V));
    cudaStream_t s = h->stream;
    Plan pl = make_plan(shape, 0, shape[0], 1, h->prof);
    StageClock clk(h);
    for (int64_t i0 = 0; i0 < n; i0 += per) {
        const int64_t nb = std::min<int64_t>(per, n - i0);
        const long long TV = V * nb;
        pl.nvol = (int)nb;
        // input -> device (always into an aligned scratch copy)
        B4D_TRY(h->in.ensure((size_t)TV * sizeof(T)));
        // one uint16 volume from host memory: uploaded in chunks behind the stage-1 matcher
        const bool stream_in = sizeof(T) == 2 && !in_dev && can_stream_upload(h, pl);
        if (!stream_in) CU_TRY(copy_in(h, h->in.p, in + i0 * V, (size_t)TV * sizeof(T), in_dev, s));
        B4D_TRY(h->u16.ensure((size_t)TV * sizeof(uint16_t) + 16));
        float *d_out = nullptr;
        if (out_dev && (reinterpret_cast<uintptr_t>(out + i0 * V) & 15) == 0) {
            d_out = out + i0 * V;
        } else {
            B4D_TRY(h->out.ensure((size_t)TV * sizeof(float)));
            d_out = h->out.as<float>();
        }
        MatchMap mm;
        float centre = 0.0f;
        float *d_zf = nullptr;
        uint16_t *d_u = h->u16.as<uint16_t>();
        clk.mark(-1, 0);
        if (sizeof(T) == 2) {
            B4D_TRY(h->zf.ensure((size_t)TV * sizeof(float)));
            if (!stream_in) B4D_TRY(convert_u16(h, h->in.as<uint16_t>(), h->zf.as<float>(), TV, &mm));
            d_zf = h->zf.as<float>();
            d_u = h->in.as<uint16_t>();  // the staged copy doubles as the matching image
        } else {
            B4D_TRY(derive_match_map(h, h->in.as<float>(), TV, sigma, &mm, &centre));
            if (centre != 0.0f) {  // large DC level: denoise z - c0 (in the scratch copy), add c0 back at the end
                b4d_launch_add_scalar(h->in.as<float>(), TV, -centre, s);
                B4D_TRY(derive_match_map(h, h->in.as<float>(), TV, sigma, &mm));
            }
            b4d_launch_to_match(h->in.as<float>(), h->u16.as<uint16_t>(), TV, mm.cf, mm.scale, mm.ishift, s);
            d_zf = h->in.as<float>();
        }
        clk.mark(B4D_T_PREP, 2);
        const bool to_host = !out_dev && nb == 1 && h->prof.stages == 2 && centre == 0.0f;
        HostSink sink{to_host ? out + i0 * V : nullptr, 0, pl.D};
        Pass ps;
        B4D_TRY(make_pass(h, pl, sigma, mm, d_zf, d_u, d_out, clk, ps));
        B4D_TRY(denoise_pass(ps, stream_in ? reinterpret_cast<const uint16_t *>(in + i0 * V) : nullptr, &sink,
                             nullptr));
        if (centre != 0.0f) b4d_launch_add_scalar(d_out, TV, centre, s);
        if (!sink.done && d_out != out + i0 * V)
            CU_TRY(copy_out(h, out + i0 * V, d_out, (size_t)TV * sizeof(float), out_dev, s));
        B4D_TRY(finish(h, clk));
    }
    return 0;
}

// The open slab of the two-call form and an owned range inside it.
int check_open_slab(const b4d_handle *h, int64_t own_begin, int64_t own_end) {
    if (!h->slab_open) return fail(B4D_ERR_INVALID, "b4d_slab_stage1_u16 has not been called");
    if (own_begin < h->slab_z_begin || own_end > h->slab_z_begin + h->slab.D || own_begin >= own_end)
        return fail(B4D_ERR_INVALID, "owned range outside the slab");
    return 0;
}
int make_slab_pass(b4d_handle *h, StageClock &clk, Pass &ps) {
    return make_pass(h, h->slab, h->slab_sigma, h->slab_mm, h->zf.as<float>(), h->in.as<uint16_t>(),
                     h->out.as<float>(), clk, ps);
}

}  // namespace

// ================================================================ C ABI =====
extern "C" {

int b4d_version(void) { return B4D_ABI_VERSION; }
const char *b4d_last_error(void) { return g_err.c_str(); }
void b4d_default_profile(b4d_profile *p) {
    if (p) default_profile(p);
}

int b4d_create(int device, const b4d_profile *profile, b4d_handle **out) {
    if (!out) return fail(B4D_ERR_INVALID, "out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(B4D_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                      " (libb4d has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return fail(B4D_ERR_INVALID, "device index out of range");
    b4d_profile prof;
    default_profile(&prof);
    if (profile) {
        prof = *profile;
        B4D_TRY(check_profile(prof));
    }
    CU_TRY(cudaSetDevice(device));
    b4d_handle *h = new b4d_handle();
    h->device = device;
    h->prof = prof;
    cudaError_t es = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (es != cudaSuccess) {
        delete h;
        return fail(B4D_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(es));
    }
    es = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
    if (es != cudaSuccess) {
        cudaStreamDestroy(h->stream);
        delete h;
        return fail(B4D_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(es));
    }
    reset_timings(h);
    std::memset(h->match_stats, 0, sizeof(h->match_stats));
    *out = h;
    return 0;
}

void b4d_destroy(b4d_handle *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    for (DevBuf *b : {&h->coh_x, &h->coh_sm, &h->coh_tmp, &h->coh_keys, &h->coh_sums, &h->coh_lab, &h->coh_w}) b->release();
    for (DevBuf *b : {&h->in, &h->u16, &h->zf, &h->numq, &h->gmap, &h->basic, &h->out, &h->widx, &h->cnt,
                      &h->ssd, &h->refs, &h->hist, &h->partial, &h->sink, &h->stats, &h->s2, &h->cells, &h->tcls,
                      &h->alt_in, &h->alt_zf, &h->alt_out, &h->alt_partial, &h->alt_sink, &h->nz_hist, &h->nz_sel,
                      &h->nz_res, &h->nz_full})
        b->release();
    if (h->pre.ev0) cudaEventDestroy(h->pre.ev0);
    if (h->pre.ev1) cudaEventDestroy(h->pre.ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    delete h;
}

int b4d_set_profile(b4d_handle *h, const b4d_profile *profile) {
    if (!h || !profile) return fail(B4D_ERR_INVALID, "NULL argument");
    B4D_TRY(check_profile(*profile));
    h->prof = *profile;
    return 0;
}

int64_t b4d_num_refs(const int64_t shape[3]) {
    if (!shape || check_shape(shape)) return -1;
    return (int64_t)ref_origins(shape[0]).size() * (int64_t)ref_origins(shape[1]).size() *
           (int64_t)ref_origins(shape[2]).size();
}

int b4d_set_pipeline_min_voxels(b4d_handle *h, int64_t voxels) {
    if (!h || voxels < 0) return fail(B4D_ERR_INVALID, "bad argument");
    h->pipeline_min_voxels = voxels;
    return 0;
}

int b4d_set_pass_voxels(b4d_handle *h, int64_t voxels) {
    if (!h || voxels < 0) return fail(B4D_ERR_INVALID, "bad argument");
    h->pass_voxels = voxels == 0 ? CHUNK_VOXELS : std::max<long long>(voxels, 4096);
    return 0;
}

// `n` uint16 volumes, each larger than a pass: z-slabs with the no-exchange halo, one after the other on this
// GPU (b4d_denoise_slab_u16); equal to the one-pass result bit for bit, like the multi-GPU slabs.  The timings
// and match statistics are summed over all slabs.
static int denoise_oversize_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3], float sigma,
                                float *out, int in_on_device, int out_on_device) {
    const int64_t D = shape[0], P = shape[1] * shape[2], V = D * P;
    const int64_t halo = (h->prof.search_ht + 2) + (h->prof.stages == 2 ? h->prof.search_wie + 2 : 0);
    const int64_t planes = h->pass_voxels / P;
    if (planes < 2 * halo + 4)
        return fail(B4D_ERR_TOO_LARGE, "a pass cannot hold two halos of this plane size: raise b4d_set_pass_voxels "
                                       "or shard the volume in y / x");
    const int64_t nslab = (D + (planes - 2 * halo) - 1) / (planes - 2 * halo);
    const int64_t own = (D + nslab - 1) / nslab;
    float t_ms[B4D_T_COUNT] = {};
    int64_t launches[B4D_T_COUNT] = {};
    unsigned long long stats[4] = {};
    for (int64_t i = 0; i < n; ++i)
        for (int64_t ob = 0; ob < D; ob += own) {
            const int64_t oe = std::min(D, ob + own), zb = std::max<int64_t>(0, ob - halo), ze = std::min(D, oe + halo);
            const int64_t sshape[3] = {ze - zb, shape[1], shape[2]};
            B4D_TRY(b4d_denoise_slab_u16(h, in + i * V + zb * P, sshape, zb, D, ob, oe, sigma, out + i * V + ob * P,
                                         in_on_device, out_on_device));
            for (int k = 0; k < B4D_T_COUNT; ++k) {
                t_ms[k] += h->t_ms[k];
                launches[k] += h->launches[k];
            }
            for (int k = 0; k < 4; ++k) stats[k] += h->match_stats[k];
        }
    std::memcpy(h->t_ms, t_ms, sizeof(t_ms));
    std::memcpy(h->launches, launches, sizeof(launches));
    std::memcpy(h->match_stats, stats, sizeof(stats));
    return 0;
}

int b4d_denoise_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3], float sigma, float *out,
                    int in_on_device, int out_on_device) {
    if (h && in && out && shape && n >= 1 && shape[0] > 0 && shape[1] > 0 && shape[2] > 0 &&
        shape[0] * shape[1] * shape[2] > h->pass_voxels) {
        B4D_TRY(common_checks(h, in, out, shape, sigma));
        return denoise_oversize_u16(h, in, n, shape, sigma, out, in_on_device, out_on_device);
    }
    return denoise_batch<uint16_t>(h, in, n, shape, sigma, out, in_on_device, out_on_device);
}
int b4d_denoise_f32(b4d_handle *h, const float *in, int64_t n, const int64_t shape[3], float sigma, float *out,
                    int in_on_device, int out_on_device) {
    return denoise_batch<float>(h, in, n, shape, sigma, out, in_on_device, out_on_device);
}

int b4d_targets_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3], const float *offsets,
                    float sigma, float max_count, float *raw_out, float *teacher_out, int in_on_device,
                    int out_on_device) {
    B4D_TRY(common_checks(h, in, teacher_out, shape, sigma));
    if (n < 1 || !offsets) return fail(B4D_ERR_INVALID, "n must be >= 1 and offsets non-NULL");
    if (h->prof.stages != 2) return fail(B4D_ERR_INVALID, "target generation needs stages = 2");
    reset_timings(h);
    const long long V = shape[0] * shape[1] * shape[2];
    int64_t per = std::max<int64_t>(1, std::min<int64_t>(n, h->pass_voxels / V));
    // With host buffers a pass is cut into four chunks on two buffer sets: while chunk c computes, the
    // teacher of chunk c - 1 and the raw of chunk c go back and chunk c + 1 comes up on the copy stream.
    if ((!in_on_device || !out_on_device) && per >= 8 && V * per >= h->pipeline_min_voxels) per = (per + 3) / 4;
    cudaStream_t s = h->stream, cs = h->copy_stream;
    Plan pl = make_plan(shape, 0, shape[0], 1, h->prof);
    StageClock clk(h);
    EventSet owned;
    DevBuf *b_in[2] = {&h->in, &h->alt_in}, *b_zf[2] = {&h->zf, &h->alt_zf}, *b_out[2] = {&h->out, &h->alt_out};
    DevBuf *b_par[2] = {&h->partial, &h->alt_partial}, *b_sink[2] = {&h->sink, &h->alt_sink};
    int64_t prev_i0 = -1, prev_nb = 0;
    int prev_set = 0;
    cudaEvent_t prev_done = nullptr;
    auto teacher_back = [&]() -> int {  // teacher of the previous chunk, once its clip has run
        if (prev_i0 < 0) return 0;
        CU_TRY(cudaStreamWaitEvent(cs, prev_done, 0));
        CU_TRY(copy_out(h, teacher_out + prev_i0 * V, b_out[prev_set]->p, (size_t)(V * prev_nb) * sizeof(float),
                        out_on_device, cs));
        return 0;
    };
    int64_t c = 0;
    for (int64_t i0 = 0; i0 < n; i0 += per, ++c) {
        const int set = (int)(c & 1);
        const int64_t nb = std::min<int64_t>(per, n - i0);
        const long long TV = V * nb;
        pl.nvol = (int)nb;
        B4D_TRY(b_in[set]->ensure((size_t)TV * sizeof(uint16_t)));
        B4D_TRY(b_zf[set]->ensure((size_t)TV * sizeof(float)));
        B4D_TRY(b_out[set]->ensure((size_t)TV * sizeof(float)));
        B4D_TRY(b_par[set]->ensure((size_t)nb * sizeof(float)));
        // copy stream: counts up, raw = float32(counts) - offset, range of the counts.  In stream order this
        // follows the copy-out of chunk c - 2, the last reader of this buffer set.
        CU_TRY(copy_in(h, b_in[set]->p, in + i0 * V, (size_t)TV * sizeof(uint16_t), in_on_device, cs));
        CU_TRY(cudaMemcpyAsync(b_par[set]->p, offsets + i0, (size_t)nb * sizeof(float), cudaMemcpyHostToDevice, cs));
        B4D_TRY(range_reset(*b_sink[set], cs));
        b4d_launch_u16_sub_offset(b_in[set]->as<uint16_t>(), b_par[set]->as<float>(), b_zf[set]->as<float>(), V, TV,
                                  b_sink[set]->as<unsigned>(), cs);
        double lo = 0, hi = 0;
        B4D_TRY(range_read(*b_sink[set], cs, &lo, &hi));
        float omin = offsets[i0], omax = offsets[i0];
        for (int64_t k = 0; k < nb; ++k) {
            omin = std::min(omin, offsets[i0 + k]);
            omax = std::max(omax, offsets[i0 + k]);
        }
        if (!std::isfinite(omin) || !std::isfinite(omax)) return fail(B4D_ERR_INVALID, "offsets must be finite");
        // Matching is invariant to a constant shift per volume: stage 1 matches on the counts themselves,
        // the stage-2 matching image rint(basic) + ishift only has to stay inside uint16.
        MatchMap mm;
        mm.ishift = centre_shift(lo - std::ceil((double)omax), hi - std::floor((double)omin));
        // compute stream: the chunk's two stages and the clip (its inputs are complete: the copy stream was
        // synchronised above)
        clk.mark(-1, 0);
        Pass ps;
        B4D_TRY(make_pass(h, pl, sigma, mm, b_zf[set]->as<float>(), b_in[set]->as<uint16_t>(),
                          b_out[set]->as<float>(), clk, ps));
        B4D_TRY(denoise_pass(ps, nullptr, nullptr, nullptr));
        b4d_launch_clip(b_out[set]->as<float>(), TV, max_count, s);
        cudaEvent_t done;
        CU_TRY(owned.make(&done));
        CU_TRY(cudaEventRecord(done, s));
        // copy stream again, while this chunk computes: teacher of the previous chunk, raw of this one
        B4D_TRY(teacher_back());
        if (raw_out)
            CU_TRY(copy_out(h, raw_out + i0 * V, b_zf[set]->p, (size_t)TV * sizeof(float), out_on_device, cs));
        prev_i0 = i0;
        prev_nb = nb;
        prev_set = set;
        prev_done = done;
    }
    B4D_TRY(teacher_back());
    CU_TRY(cudaStreamSynchronize(cs));
    return finish(h, clk);
}

static int denoise_slab_impl(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                             int64_t z_total, int64_t own_begin, int64_t own_end, float sigma, void *out,
                             int in_on_device, int out_on_device, const QuantSpec *q) {
    B4D_TRY(common_checks(h, in, out, shape, sigma));
    if (q && h->prof.stages != 2) return fail(B4D_ERR_INVALID, "quantized output needs stages = 2");
    if (q && !(q->step >= 1.0f)) return fail(B4D_ERR_INVALID, "step must be >= 1");
    const size_t esz = q ? sizeof(uint16_t) : sizeof(float);
    if (z_begin < 0 || z_begin + shape[0] > z_total || own_begin < z_begin || own_end > z_begin + shape[0] ||
        own_begin >= own_end)
        return fail(B4D_ERR_INVALID, "slab / owned range inconsistent");
    reset_timings(h);
    const long long P = shape[1] * shape[2];
    const Plan pl = make_plan(shape, z_begin, z_total, 1, h->prof);
    StageClock clk(h);
    MatchMap mm;
    const uint16_t *host_src = nullptr;
    B4D_TRY(stage_u16_input(h, pl, in, in_on_device, clk, &mm, &host_src));
    HostSink sink{out_on_device ? nullptr : out, own_begin - z_begin, own_end - z_begin};
    Pass ps;
    B4D_TRY(make_pass(h, pl, sigma, mm, h->zf.as<float>(), h->in.as<uint16_t>(), h->out.as<float>(), clk, ps));
    B4D_TRY(denoise_pass(ps, host_src, &sink, q));
    if (!sink.done)
        CU_TRY(copy_out(h, out, h->out.as<char>() + (size_t)sink.p0 * P * esz, (size_t)(sink.p1 - sink.p0) * P * esz,
                        out_on_device, h->stream));
    return finish(h, clk);
}
int b4d_denoise_slab_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                         int64_t z_total, int64_t own_begin, int64_t own_end, float sigma, float *out,
                         int in_on_device, int out_on_device) {
    return denoise_slab_impl(h, in, shape, z_begin, z_total, own_begin, own_end, sigma, out, in_on_device,
                             out_on_device, nullptr);
}
int b4d_denoise_slab_q16_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin,
                             int64_t z_total, int64_t own_begin, int64_t own_end, float sigma, float offset_sub,
                             float offset_add, float step, int truncate, uint16_t *out, int in_on_device,
                             int out_on_device) {
    const QuantSpec q{offset_sub, offset_add, step, truncate};
    return denoise_slab_impl(h, in, shape, z_begin, z_total, own_begin, own_end, sigma, out, in_on_device,
                             out_on_device, &q);
}
int b4d_denoise_q16_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], float sigma, float offset_sub,
                        float offset_add, float step, int truncate, uint16_t *out, int in_on_device,
                        int out_on_device) {
    if (!shape) return fail(B4D_ERR_INVALID, "NULL argument");
    return b4d_denoise_slab_q16_u16(h, in, shape, 0, shape[0], 0, shape[0], sigma, offset_sub, offset_add, step,
                                    truncate, out, in_on_device, out_on_device);
}

int b4d_slab_stage1_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], int64_t z_begin, int64_t z_total,
                        float sigma, int in_on_device) {
    B4D_TRY(common_checks(h, in, in, shape, sigma));
    if (z_begin < 0 || z_begin + shape[0] > z_total) return fail(B4D_ERR_INVALID, "slab range inconsistent");
    if (h->prof.stages != 2) return fail(B4D_ERR_INVALID, "the two-call slab form needs stages = 2");
    reset_timings(h);
    h->slab_open = false;
    h->slab = make_plan(shape, z_begin, z_total, 1, h->prof);
    h->slab_z_begin = z_begin;
    h->slab_sigma = sigma;
    StageClock clk(h);
    MatchMap mm;
    const uint16_t *host_src = nullptr;
    B4D_TRY(stage_u16_input(h, h->slab, in, in_on_device, clk, &mm, &host_src));
    Pass ps;
    B4D_TRY(make_pass(h, h->slab, sigma, mm, h->zf.as<float>(), h->in.as<uint16_t>(), h->out.as<float>(), clk, ps));
    B4D_TRY(stage1(ps, host_src, false));
    CU_TRY(cudaStreamSynchronize(h->stream));
    clk.resolve();
    h->pre.done = false;
    h->slab_mm = ps.mm;
    h->slab_open = true;
    return 0;
}

int b4d_slab_basic_planes(b4d_handle *h, int64_t plane0, int64_t nplanes, float *buf, int to_handle,
                          int buf_on_device) {
    if (!h || !buf) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!h->slab_open) return fail(B4D_ERR_INVALID, "b4d_slab_stage1_u16 has not been called");
    if (plane0 < 0 || nplanes < 0 || plane0 + nplanes > h->slab.D)
        return fail(B4D_ERR_INVALID, "plane range outside the slab");
    CU_TRY(cudaSetDevice(h->device));
    const size_t P = (size_t)h->slab.H * h->slab.W;
    float *dev = h->basic.as<float>() + (size_t)plane0 * P;
    const size_t bytes = (size_t)nplanes * P * sizeof(float);
    if (to_handle)
        CU_TRY(copy_in(h, dev, buf, bytes, buf_on_device, h->stream));
    else
        CU_TRY(copy_out(h, buf, dev, bytes, buf_on_device, h->stream));
    CU_TRY(cudaStreamSynchronize(h->stream));
    return 0;
}

static int slab_stage2_impl(b4d_handle *h, int64_t own_begin, int64_t own_end, void *out, int out_on_device,
                            const QuantSpec *q) {
    if (!h || !out) return fail(B4D_ERR_INVALID, "NULL argument");
    if (q && !(q->step >= 1.0f)) return fail(B4D_ERR_INVALID, "step must be >= 1");
    const size_t esz = q ? sizeof(uint16_t) : sizeof(float);
    B4D_TRY(check_open_slab(h, own_begin, own_end));
    CU_TRY(cudaSetDevice(h->device));
    const long long P = (long long)h->slab.H * h->slab.W;
    const bool had_pre = h->pre.done;
    StageClock clk(h);
    clk.mark(-1, 0);
    HostSink sink{out_on_device ? nullptr : out, own_begin - h->slab_z_begin, own_end - h->slab_z_begin};
    Pass ps;
    B4D_TRY(make_slab_pass(h, clk, ps));
    B4D_TRY(had_pre ? stage2_front_rest(ps) : stage2_front_whole(ps, false));
    B4D_TRY(stage2_back(ps, &sink, q));
    if (!sink.done)
        CU_TRY(copy_out(h, out, h->out.as<char>() + (size_t)sink.p0 * P * esz, (size_t)(sink.p1 - sink.p0) * P * esz,
                        out_on_device, h->stream));
    B4D_TRY(finish(h, clk));
    if (had_pre) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->pre.ev0, h->pre.ev1) == cudaSuccess) {
            h->t_ms[B4D_T_MATCH2] += ms;
            h->launches[B4D_T_MATCH2] += 5;
        } else {
            cudaGetLastError();
        }
    }
    h->slab_open = false;
    return 0;
}
int b4d_slab_stage2(b4d_handle *h, int64_t own_begin, int64_t own_end, float *out, int out_on_device) {
    return slab_stage2_impl(h, own_begin, own_end, out, out_on_device, nullptr);
}
int b4d_slab_stage2_q16(b4d_handle *h, int64_t own_begin, int64_t own_end, float offset_sub, float offset_add,
                        float step, int truncate, uint16_t *out, int out_on_device) {
    const QuantSpec q{offset_sub, offset_add, step, truncate};
    return slab_stage2_impl(h, own_begin, own_end, out, out_on_device, &q);
}

float *b4d_slab_basic_ptr(b4d_handle *h) {
    if (!h || !h->slab_open) {
        fail(B4D_ERR_INVALID, "b4d_slab_stage1_u16 has not been called");
        return nullptr;
    }
    return h->basic.as<float>();
}

int b4d_slab_stage2_begin(b4d_handle *h, int64_t own_begin, int64_t own_end) {
    if (!h) return fail(B4D_ERR_INVALID, "NULL argument");
    B4D_TRY(check_open_slab(h, own_begin, own_end));
    CU_TRY(cudaSetDevice(h->device));
    StageClock clk(h);
    clk.mark(-1, 0);
    if (!h->pre.ev0) {
        CU_TRY(cudaEventCreate(&h->pre.ev0));
        CU_TRY(cudaEventCreate(&h->pre.ev1));
    }
    CU_TRY(cudaEventRecord(h->pre.ev0, h->stream));
    Pass ps;
    B4D_TRY(make_slab_pass(h, clk, ps));
    B4D_TRY(stage2_front_owned(ps, (int)(own_begin - h->slab_z_begin), (int)(own_end - h->slab_z_begin)));
    CU_TRY(cudaEventRecord(h->pre.ev1, h->stream));
    return 0;  // no synchronisation: the launches run while the caller exchanges planes
}

int b4d_match_stage1(b4d_handle *h, const uint16_t *in, const int64_t shape[3], float sigma, int32_t *idx,
                     uint64_t *ssd, int32_t *count) {
    if (!idx || !ssd || !count) return fail(B4D_ERR_INVALID, "NULL argument");
    B4D_TRY(common_checks(h, in, idx, shape, sigma));
    const int64_t Dc = shape[0] - L + 1, Hc = shape[1] - L + 1, Wc = shape[2] - L + 1;
    if (Dc * Hc * Wc > INT32_MAX) return fail(B4D_ERR_TOO_LARGE, "candidate index space exceeds int32");
    const b4d_profile &p = h->prof;
    cudaStream_t s = h->stream;
    reset_timings(h);
    const Plan pl = make_plan(shape, 0, shape[0], 1, p);
    B4dGeom g, g_unused;
    B4D_TRY(upload_geometry(h, pl, &g, &g_unused));
    const long long V = shape[0] * shape[1] * shape[2];
    B4D_TRY(h->u16.ensure((size_t)V * sizeof(uint16_t) + 16));
    CU_TRY(cudaMemcpyAsync(h->u16.p, in, (size_t)V * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
    const long long R = g.refs_per_vol;
    const int K = p.k_ht, Ns = p.search_ht, r = Ns / 2;
    B4D_TRY(h->widx.ensure((size_t)R * std::max(p.k_ht, p.k_wie) * sizeof(uint16_t)));
    B4D_TRY(h->cnt.ensure((size_t)R));
    B4D_TRY(h->ssd.ensure((size_t)R * K * sizeof(uint32_t)));
    B4D_TRY(h->stats.ensure(4 * sizeof(unsigned long long)));
    CU_TRY(cudaMemsetAsync(h->stats.p, 0, 4 * sizeof(unsigned long long), s));
    B4D_TRY(h->s2.ensure((size_t)V * sizeof(uint2)));
    B4D_TRY(h->cells.ensure((size_t)pl.D * g.ty * g.tx * sizeof(uint32_t)));
    B4D_TRY(h->tcls.ensure((size_t)g.tz * g.ty * g.tx * sizeof(uint32_t)));
    b4d_launch_block_energy(h->u16.as<uint16_t>(), h->s2.as<uint2>(), pl.D, pl.H, pl.W, 1, s);
    MatchParams mp;
    mp.g = g;
    mp.u = h->u16.as<uint16_t>();
    mp.s21 = h->s2.as<uint2>();
    mp.cells = h->cells.as<uint32_t>();
    mp.tcls = h->tcls.as<uint32_t>();
    B4D_TRY(tau_for(p.tau_ht, sigma, 1.0f, Ns, &mp.tau));
    mp.K = K;
    mp.widx = h->widx.as<uint16_t>();
    mp.cnt = h->cnt.as<uint8_t>();
    mp.ssd_out = h->ssd.as<uint32_t>();
    mp.stats = h->stats.as<unsigned long long>();
    StageClock clk(h);
    clk.mark(-1, 0);
    b4d_launch_match(mp, Ns, s);
    clk.mark(B4D_T_MATCH1, 4);
    CU_TRY(cudaGetLastError());
    std::vector<uint16_t> hw((size_t)R * K);
    std::vector<uint32_t> hs((size_t)R * K);
    std::vector<uint8_t> hc((size_t)R);
    CU_TRY(cudaMemcpyAsync(hw.data(), mp.widx, hw.size() * sizeof(uint16_t), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaMemcpyAsync(hs.data(), mp.ssd_out, hs.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaMemcpyAsync(hc.data(), mp.cnt, hc.size(), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaMemcpyAsync(h->match_stats, h->stats.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    clk.resolve();
    const int nry = g.nry, nrx = g.nrx;
    for (long long ri = 0; ri < R; ++ri) {
        const int oz = pl.rz1[ri / ((long long)nry * nrx)], oy = pl.ry[(ri / nrx) % nry], ox = pl.rx[ri % nrx];
        count[ri] = hc[ri];
        for (int k = 0; k < K; ++k) {
            if (k < hc[ri]) {
                const int wi = hw[ri * K + k];
                const int cz = oz - r + wi / (Ns * Ns), cy = oy - r + (wi / Ns) % Ns, cx = ox - r + wi % Ns;
                idx[ri * K + k] = (int32_t)(((int64_t)cz * Hc + cy) * Wc + cx);
                ssd[ri * K + k] = hs[ri * K + k];
            } else {
                idx[ri * K + k] = -1;
                ssd[ri * K + k] = UINT64_MAX;
            }
        }
    }
    return 0;
}

static int quantize_impl(b4d_handle *h, const float *in, int64_t n, float offset_sub, float offset_add, float step,
                         uint16_t *out, int in_on_device, int out_on_device, bool trunc) {
    if (!h || !in || !out || n < 0) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!(step >= 1.0f)) return fail(B4D_ERR_INVALID, "step must be >= 1");
    CU_TRY(cudaSetDevice(h->device));
    if (n == 0) return 0;
    cudaStream_t s = h->stream;
    const float *d_in = in;
    uint16_t *d_out = out;
    if (!in_on_device || (reinterpret_cast<uintptr_t>(in) & 15)) {
        B4D_TRY(h->in.ensure((size_t)n * sizeof(float)));
        CU_TRY(copy_in(h, h->in.p, in, (size_t)n * sizeof(float), in_on_device, s));
        d_in = h->in.as<float>();
    }
    if (!out_on_device || (reinterpret_cast<uintptr_t>(out) & 15)) {
        B4D_TRY(h->u16.ensure((size_t)n * sizeof(uint16_t) + 16));
        d_out = h->u16.as<uint16_t>();
    }
    if (trunc) b4d_launch_quantize_trunc(d_in, d_out, n, offset_sub, offset_add, step, s);
    else b4d_launch_quantize(d_in, d_out, n, offset_sub, offset_add, step, s);
    CU_TRY(cudaGetLastError());
    if (d_out != out)
        CU_TRY(copy_out(h, out, d_out, (size_t)n * sizeof(uint16_t), out_on_device, s));
    CU_TRY(cudaStreamSynchronize(s));
    return 0;
}
int b4d_quantize_u16(b4d_handle *h, const float *in, int64_t n, float offset_sub, float offset_add, float step,
                     uint16_t *out, int in_on_device, int out_on_device) {
    return quantize_impl(h, in, n, offset_sub, offset_add, step, out, in_on_device, out_on_device, false);
}
int b4d_quantize_trunc_u16(b4d_handle *h, const float *in, int64_t n, float offset_sub, float offset_add, float step,
                           uint16_t *out, int in_on_device, int out_on_device) {
    return quantize_impl(h, in, n, offset_sub, offset_add, step, out, in_on_device, out_on_device, true);
}

// Exact NumPy-2 semantics on float32 data (float32 virtual index, float32 lerp):
//   q = float32(pct) / float32(100); vi = float32(n - 1) * q;  lerp in float32.
static float percentile_f32(const std::vector<unsigned long long> &hist, int first_bin, long long n, double pct) {
    auto order_stat = [&](long long k) -> float {  // k-th smallest (0-based) among bins >= first_bin
        long long c = 0;
        for (int v = first_bin; v < 65536; ++v) {
            c += (long long)hist[v];
            if (k < c) return (float)v;
        }
        return 65535.0f;
    };
    volatile float q = (float)pct / 100.0f;
    volatile float vi = (float)(n - 1) * q;
    long long pi, ni;
    const float prev = std::floor(vi);
    if (vi >= (float)(n - 1)) {
        pi = ni = n - 1;
    } else if (vi < 0) {
        pi = ni = 0;
    } else {
        pi = (long long)prev;
        ni = pi + 1;
    }
    volatile float g = vi - prev;
    const float a = order_stat(pi), b = order_stat(ni);
    volatile float d = b - a;
    volatile float dg = d * g;
    volatile float r = a + dg;
    if (g >= 0.5f) {
        volatile float omg = 1.0f - g;
        volatile float t = d * omg;
        r = b - t;
    }
    return r;
}

// Threshold of make_foreground_mask (metrics.py:54-58) for raw = float32(u) - off, from the exact histogram of
// u.  Order statistics commute with the monotone map u -> float32(u) - off, so every float32 step of the NumPy
// code (median = mean of the two middle values, |raw - med|, its median, + 1e-6, * 1.4826, med + k * sigma;
// Python-float constants are weak under NEP 50, the arithmetic stays float32) is reproduced on the
// distinct values only.
static float robust_threshold(const unsigned long long *hist, long long n, float off, float k) {
    auto kth_u = [&](long long r) -> int {
        long long c = 0;
        for (int v = 0; v < 65536; ++v) {
            c += (long long)hist[v];
            if (r < c) return v;
        }
        return 65535;
    };
    const float a = (float)kth_u((n - 1) / 2) - off, b = (float)kth_u(n / 2) - off;
    const float med = (a + b) / 2.0f;
    std::vector<std::pair<float, unsigned long long>> dev;
    for (int v = 0; v < 65536; ++v)
        if (hist[v]) dev.emplace_back(std::fabs(((float)v - off) - med), hist[v]);
    std::sort(dev.begin(), dev.end());
    auto kth_d = [&](long long r) -> float {
        long long c = 0;
        for (const auto &e : dev) {
            c += (long long)e.second;
            if (r < c) return e.first;
        }
        return dev.back().first;
    };
    const float mad = (kth_d((n - 1) / 2) + kth_d(n / 2)) / 2.0f + 1e-6f;
    const float sigma = 1.4826f * mad;
    return med + k * sigma;
}

int b4d_foreground_mask_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3],
                            const float *offsets, float k, int dilate, uint8_t *out, int in_on_device,
                            int out_on_device) {
    if (!h || !in || !out || !shape || !offsets) return fail(B4D_ERR_INVALID, "NULL argument");
    if (n < 1) return fail(B4D_ERR_INVALID, "n must be >= 1");
    for (int a = 0; a < 3; ++a)
        if (shape[a] < 1 || shape[a] > INT32_MAX) return fail(B4D_ERR_INVALID, "bad shape");
    if (dilate < 0 || dilate > 8) return fail(B4D_ERR_INVALID, "dilate must be in [0, 8]");
    if (!std::isfinite(k)) return fail(B4D_ERR_INVALID, "k must be finite");
    const long long V = shape[0] * shape[1] * shape[2];
    if (V > INT32_MAX) return fail(B4D_ERR_TOO_LARGE, "a patch may hold at most 2^31 - 1 voxels");
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    constexpr int G = 32;  // patches per histogram round trip
    const int64_t per = std::max<int64_t>(1, std::min<int64_t>(n, h->pass_voxels / V));
    std::vector<unsigned long long> hist((size_t)G * 65536);
    for (int64_t i0 = 0; i0 < n; i0 += per) {
        const int64_t nb = std::min<int64_t>(per, n - i0);
        const long long TV = V * nb;
        const uint16_t *d_in = in + i0 * V;
        if (!in_on_device) {
            B4D_TRY(h->in.ensure((size_t)TV * sizeof(uint16_t)));
            CU_TRY(copy_in(h, h->in.p, in + i0 * V, (size_t)TV * sizeof(uint16_t), 0, s));
            d_in = h->in.as<uint16_t>();
        }
        std::vector<float> thr((size_t)nb);
        B4D_TRY(h->hist.ensure((size_t)G * 65536 * sizeof(unsigned long long)));
        for (int64_t g0 = 0; g0 < nb; g0 += G) {
            const int64_t ng = std::min<int64_t>(G, nb - g0);
            CU_TRY(cudaMemsetAsync(h->hist.p, 0, (size_t)ng * 65536 * sizeof(unsigned long long), s));
            for (int64_t g = 0; g < ng; ++g)
                b4d_launch_hist(d_in + (g0 + g) * V, V, h->hist.as<unsigned long long>() + g * 65536, s);
            CU_TRY(cudaGetLastError());
            CU_TRY(copy_out(h, hist.data(), h->hist.p, (size_t)ng * 65536 * sizeof(unsigned long long), 0, s));
            CU_TRY(cudaStreamSynchronize(s));
            for (int64_t g = 0; g < ng; ++g) {
                if (!std::isfinite(offsets[i0 + g0 + g])) return fail(B4D_ERR_INVALID, "offsets must be finite");
                thr[(size_t)(g0 + g)] = robust_threshold(hist.data() + g * 65536, V, offsets[i0 + g0 + g], k);
            }
        }
        B4D_TRY(h->partial.ensure((size_t)nb * 2 * sizeof(float)));
        float *d_off = h->partial.as<float>(), *d_thr = d_off + nb;
        CU_TRY(cudaMemcpyAsync(d_off, offsets + i0, (size_t)nb * sizeof(float), cudaMemcpyHostToDevice, s));
        CU_TRY(cudaMemcpyAsync(d_thr, thr.data(), (size_t)nb * sizeof(float), cudaMemcpyHostToDevice, s));
        uint8_t *d_out = out + i0 * V;
        if (!out_on_device) {
            B4D_TRY(h->u16.ensure((size_t)TV + 16));
            d_out = h->u16.as<uint8_t>();
        }
        b4d_launch_fg_mask(d_in, d_off, d_thr, (int)shape[0], (int)shape[1], (int)shape[2], TV, dilate, d_out, s);
        CU_TRY(cudaGetLastError());
        if (!out_on_device) CU_TRY(copy_out(h, out + i0 * V, d_out, (size_t)TV, 0, s));
        CU_TRY(cudaStreamSynchronize(s));  // thr / offsets staging is reused by the next chunk
    }
    return 0;
}

int b4d_chunk_shuffle_u16(b4d_handle *h, const uint16_t *in, const int64_t shape[3], const int64_t chunk[3],
                          uint8_t *out, uint32_t *hist, int in_on_device, int out_on_device) {
    if (!h || !in || !shape || !chunk) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!out && !hist) return fail(B4D_ERR_INVALID, "nothing to compute: out and hist are both NULL");
    for (int a = 0; a < 3; ++a) {
        if (shape[a] < 1 || shape[a] > INT32_MAX) return fail(B4D_ERR_INVALID, "bad shape");
        if (chunk[a] < 1 || chunk[a] > INT32_MAX) return fail(B4D_ERR_INVALID, "bad chunk shape");
    }
    {
        double pv = 1.0;  // voxels of the largest piece
        for (int a = 0; a < 3; ++a) pv *= (double)std::min(chunk[a], shape[a]);
        if (pv > 1073741824.0) return fail(B4D_ERR_TOO_LARGE, "a piece may hold at most 2^30 voxels");
    }
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const long long n = shape[0] * shape[1] * shape[2];
    long long nchunks = 1;
    for (int a = 0; a < 3; ++a) nchunks *= (shape[a] + chunk[a] - 1) / chunk[a];
    const uint16_t *d_in = in;
    if (!in_on_device) {
        B4D_TRY(h->in.ensure((size_t)n * sizeof(uint16_t)));
        CU_TRY(copy_in(h, h->in.p, in, (size_t)n * sizeof(uint16_t), 0, s));
        d_in = h->in.as<uint16_t>();
    }
    uint8_t *d_out = out;
    if (out && !out_on_device) {
        B4D_TRY(h->u16.ensure((size_t)n * sizeof(uint16_t) + 16));
        d_out = h->u16.as<uint8_t>();
    }
    uint32_t *d_hist = hist;
    if (hist && !out_on_device) {
        B4D_TRY(h->hist.ensure((size_t)nchunks * 512 * sizeof(uint32_t)));
        d_hist = h->hist.as<uint32_t>();
    }
    b4d_launch_chunk_shuffle(d_in, (int)shape[0], (int)shape[1], (int)shape[2], (int)chunk[0], (int)chunk[1],
                             (int)chunk[2], d_out, d_hist, s);
    CU_TRY(cudaGetLastError());
    if (out && d_out != out) CU_TRY(copy_out(h, out, d_out, (size_t)n * sizeof(uint16_t), 0, s));
    if (hist && d_hist != hist) CU_TRY(copy_out(h, hist, d_hist, (size_t)nchunks * 512 * sizeof(uint32_t), 0, s));
    CU_TRY(cudaStreamSynchronize(s));
    return 0;
}

static int stats_of_hist(const std::vector<unsigned long long> &hist, int64_t n, double pct, b4d_stats *out) {
    std::memset(out, 0, sizeof(*out));
    out->n = n;
    out->n_nonzero = n - (int64_t)hist[0];
    int vmin = 65535, vmax = 0;
    for (int v = 0; v < 65536; ++v)
        if (hist[v]) {
            vmin = std::min(vmin, v);
            vmax = std::max(vmax, v);
        }
    out->vmin = vmin;
    out->vmax = vmax;
    // transforms.py:433-438: zeros are ignored unless every voxel is zero
    if (out->n_nonzero > 0) out->offset = (double)percentile_f32(hist, 1, out->n_nonzero, pct);
    else out->offset = (double)percentile_f32(hist, 0, n, pct);
    // metrics.py:55-57 in float32
    auto kth = [&](const std::vector<unsigned long long> &hh, long long k) -> long long {
        long long c = 0;
        for (size_t v = 0; v < hh.size(); ++v) {
            c += (long long)hh[v];
            if (k < c) return (long long)v;
        }
        return (long long)hh.size() - 1;
    };
    // median: mean of the two middle order statistics (equal when n is odd)
    const long long m_lo = kth(hist, (n - 1) / 2), m_hi = kth(hist, n / 2);
    const float med = ((float)m_lo + (float)m_hi) * 0.5f;  // exact: integers < 2^17
    // |x - med| in half-counts: t = |2x - (m_lo + m_hi)|
    const long long m2 = m_lo + m_hi;
    std::vector<unsigned long long> h2(131072, 0ull);
    for (int v = 0; v < 65536; ++v)
        if (hist[v]) h2[(size_t)std::llabs(2ll * v - m2)] += hist[v];
    const long long a_lo = kth(h2, (n - 1) / 2), a_hi = kth(h2, n / 2);
    const float mad_med = ((float)a_lo * 0.5f + (float)a_hi * 0.5f) * 0.5f;  // exact (quarter counts)
    volatile float mad = mad_med + 1e-6f;
    volatile float sig = 1.4826f * mad;
    out->median = med;
    out->mad = mad;
    out->sigma = sig;
    return 0;
}

int b4d_tile_stats(b4d_handle *h, const uint16_t *in, int64_t n, double pct, b4d_stats *out, int64_t *hist_out,
                   int in_on_device) {
    if (!h || !in || !out || n < 1) return fail(B4D_ERR_INVALID, "NULL argument or empty tile");
    if (!(pct >= 0.0 && pct <= 100.0)) return fail(B4D_ERR_INVALID, "percentile must be in [0, 100]");
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const uint16_t *d_in = in;
    if (!in_on_device || (reinterpret_cast<uintptr_t>(in) & 15)) {
        B4D_TRY(h->in.ensure((size_t)n * sizeof(uint16_t)));
        CU_TRY(copy_in(h, h->in.p, in, (size_t)n * sizeof(uint16_t), in_on_device, s));
        d_in = h->in.as<uint16_t>();
    }
    B4D_TRY(h->hist.ensure(65536 * sizeof(unsigned long long)));
    CU_TRY(cudaMemsetAsync(h->hist.p, 0, 65536 * sizeof(unsigned long long), s));
    b4d_launch_hist(d_in, n, h->hist.as<unsigned long long>(), s);
    CU_TRY(cudaGetLastError());
    std::vector<unsigned long long> hist(65536);
    CU_TRY(cudaMemcpyAsync(hist.data(), h->hist.p, 65536 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    if (hist_out)
        for (int v = 0; v < 65536; ++v) hist_out[v] = (int64_t)hist[v];

    return stats_of_hist(hist, n, pct, out);
}

// The statistics of an exact 65 536-bin histogram (any number of merged tiles): what b4d_tile_stats evaluates
// after its counting kernel; host arithmetic only.  Ranks that all-gather their histograms call it on the sum.
int b4d_stats_from_hist(const int64_t *hist_in, double pct, b4d_stats *out) {
    if (!hist_in || !out) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!(pct >= 0.0 && pct <= 100.0)) return fail(B4D_ERR_INVALID, "percentile must be in [0, 100]");
    std::vector<unsigned long long> hist(65536);
    long long n = 0;
    for (int v = 0; v < 65536; ++v) {
        if (hist_in[v] < 0) return fail(B4D_ERR_INVALID, "negative count");
        hist[v] = (unsigned long long)hist_in[v];
        n += hist_in[v];
    }
    if (n < 1) return fail(B4D_ERR_INVALID, "empty histogram");
    return stats_of_hist(hist, n, pct, out);
}

// DESIGN §3.11: from the two middle order statistics a <= b of |d| over m cells, in this order in float64 so that
// the result equals np.median(|d|) / (np.sqrt(8.0) * 0.6744897501960817) bit for bit.
static void noise_of_order_stats(int64_t a, int64_t b, int64_t m, double *sigma, double *mad, int64_t *cells) {
    *cells = m;
    if (m == 0) {
        *mad = *sigma = std::nan("");
        return;
    }
    *mad = ((double)a + (double)b) / 2.0;
    *sigma = *mad / (std::sqrt(8.0) * 0.6744897501960817);
}

int b4d_noise_sigma_u16(b4d_handle *h, const uint16_t *in, int64_t n, const int64_t shape[3], const int64_t tile[3],
                        double *sigma, double *mad, int64_t *cells, int64_t *hist_out, int in_on_device) {
    if (!h || !in || !shape || !sigma || !mad || !cells || n < 1) return fail(B4D_ERR_INVALID, "NULL argument or n < 1");
    B4D_TRY(check_shape(shape));
    int64_t side[3];  // tile sides in voxels; one tile per volume: the shape rounded up to even
    for (int a = 0; a < 3; ++a) {
        if (tile && (tile[a] < 2 || (tile[a] & 1))) return fail(B4D_ERR_INVALID, "tile sides must be even and >= 2");
        side[a] = tile ? tile[a] : shape[a] + (shape[a] & 1);
    }
    const int64_t vox = shape[0] * shape[1] * shape[2];
    if (n > (INT64_MAX / 2) / vox) return fail(B4D_ERR_TOO_LARGE, "input too large");
    NoiseGeom g{};
    g.vol_stride = vox;
    g.H = (int)shape[1];
    g.W = (int)shape[2];
    int nc[3], tc[3], nt[3];
    for (int a = 0; a < 3; ++a) {
        nc[a] = (int)(shape[a] / 2);
        nt[a] = side[a] >= shape[a] ? 1 : (int)((shape[a] + side[a] - 1) / side[a]);
        tc[a] = (int)std::min<int64_t>(side[a] / 2, nc[a]);  // a tile wider than the volume is the one tile
    }
    g.ncz = nc[0], g.ncy = nc[1], g.ncx = nc[2];
    g.tcz = tc[0], g.tcy = tc[1], g.tcx = tc[2];
    g.ntz = nt[0], g.nty = nt[1], g.ntx = nt[2];
    if ((int64_t)tc[0] * tc[1] * tc[2] > (int64_t)UINT32_MAX)
        return fail(B4D_ERR_TOO_LARGE, "a tile may hold at most 2^32 - 1 cells (32-bit counts)");
    // launch shape: a CTA takes about 4096 cells of one tile, as whole cell rows
    const int max_rows = tc[0] * tc[1];
    g.rows_per_cta = std::max(1, std::min(max_rows, 4096 / tc[2]));
    g.warps = std::min(8, g.rows_per_cta);
    g.ctas_per_tile = (max_rows + g.rows_per_cta - 1) / g.rows_per_cta;
    const long long ntiles = n * (long long)nt[0] * nt[1] * nt[2];
    // tiles per launch: bounds the scratch (4 KB per tile) and the grid
    const long long group = std::min<long long>(ntiles, std::min<long long>(1 << 16, INT32_MAX / g.ctas_per_tile));

    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    g.in = in;
    if (!in_on_device) {
        B4D_TRY(h->in.ensure((size_t)(n * vox) * sizeof(uint16_t)));
        CU_TRY(copy_in(h, h->in.p, in, (size_t)(n * vox) * sizeof(uint16_t), 0, s));
        g.in = h->in.as<uint16_t>();
    }
    B4D_TRY(h->nz_hist.ensure((size_t)group * 1024 * sizeof(uint32_t)));
    B4D_TRY(h->nz_sel.ensure((size_t)group * 5 * sizeof(uint32_t)));
    B4D_TRY(h->nz_res.ensure((size_t)ntiles * 3 * sizeof(uint32_t)));
    uint32_t *d_hist = h->nz_hist.as<uint32_t>(), *d_sel = h->nz_sel.as<uint32_t>();
    for (long long t0 = 0; t0 < ntiles; t0 += group) {
        const long long cnt = std::min(group, ntiles - t0);
        g.tile0 = t0;
        CU_TRY(cudaMemsetAsync(d_hist, 0, (size_t)cnt * 1024 * sizeof(uint32_t), s));
        b4d_launch_noise_pass(g, 1, cnt, d_hist, nullptr, s);
        b4d_launch_noise_select(1, d_hist, d_sel, nullptr, cnt, s);
        CU_TRY(cudaMemsetAsync(d_hist, 0, (size_t)cnt * 1024 * sizeof(uint32_t), s));
        b4d_launch_noise_pass(g, 2, cnt, d_hist, d_sel, s);
        b4d_launch_noise_select(2, d_hist, d_sel, h->nz_res.as<uint32_t>() + t0 * 3, cnt, s);
        CU_TRY(cudaGetLastError());
    }
    std::vector<unsigned long long> full;
    if (hist_out) {
        B4D_TRY(h->nz_full.ensure(B4D_NOISE_HIST_BINS * sizeof(unsigned long long)));
        CU_TRY(cudaMemsetAsync(h->nz_full.p, 0, B4D_NOISE_HIST_BINS * sizeof(unsigned long long), s));
        b4d_launch_noise_hist(g, n, h->nz_full.as<unsigned long long>(), s);
        CU_TRY(cudaGetLastError());
        full.resize(B4D_NOISE_HIST_BINS);
        CU_TRY(cudaMemcpyAsync(full.data(), h->nz_full.p, B4D_NOISE_HIST_BINS * sizeof(unsigned long long),
                               cudaMemcpyDeviceToHost, s));
    }
    std::vector<uint32_t> res((size_t)ntiles * 3);
    CU_TRY(cudaMemcpyAsync(res.data(), h->nz_res.p, res.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    for (long long t = 0; t < ntiles; ++t)
        noise_of_order_stats(res[3 * t], res[3 * t + 1], res[3 * t + 2], sigma + t, mad + t, cells + t);
    if (hist_out)
        for (int v = 0; v < B4D_NOISE_HIST_BINS; ++v) hist_out[v] = (int64_t)full[v];
    return 0;
}

// The statistics of an exact |d| histogram (any sum of per-call or per-slab histograms); host arithmetic only.
int b4d_noise_sigma_from_hist(const int64_t *hist, double *sigma, double *mad, int64_t *cells) {
    if (!hist || !sigma || !mad || !cells) return fail(B4D_ERR_INVALID, "NULL argument");
    int64_t m = 0;
    for (int v = 0; v < B4D_NOISE_HIST_BINS; ++v) {
        if (hist[v] < 0) return fail(B4D_ERR_INVALID, "negative count");
        m += hist[v];
    }
    int64_t ab[2] = {0, 0};
    const int64_t rank[2] = {(m - 1) / 2, m / 2};
    for (int k = 0; k < 2 && m > 0; ++k) {
        int64_t c = 0;
        int v = 0;
        while (c + hist[v] <= rank[k]) c += hist[v++];
        ab[k] = v;
    }
    noise_of_order_stats(ab[0], ab[1], m, sigma, mad, cells);
    return 0;
}

int b4d_last_timings(b4d_handle *h, float ms[B4D_T_COUNT], int64_t launches[B4D_T_COUNT]) {
    if (!h || !ms) return fail(B4D_ERR_INVALID, "NULL argument");
    for (int i = 0; i < B4D_T_COUNT; ++i) {
        ms[i] = h->t_ms[i];
        if (launches) launches[i] = h->launches[i];
    }
    return 0;
}

void *b4d_stream(b4d_handle *h) { return h ? (void *)h->stream : nullptr; }

// oracle-free diagnostics: [0] survivor-list retries, [1] wide (uint64) tiles, [2] slow refs, [3] byte tiles
int b4d_last_match_stats(b4d_handle *h, uint64_t out[4]) {
    if (!h || !out) return fail(B4D_ERR_INVALID, "NULL argument");
    for (int i = 0; i < 4; ++i) out[i] = h->match_stats[i];
    return 0;
}

int b4d_set_noise_model(b4d_handle *h, const float *nu_ht, const float *nu_wie) {
    if (!h) return fail(B4D_ERR_INVALID, "NULL argument");
    if (!nu_ht && !nu_wie) {
        h->psd = false;
        return 0;
    }
    if (!nu_ht || !nu_wie) return fail(B4D_ERR_INVALID, "both tables or none");
    for (int c = 0; c < 64; ++c)
        if (!(nu_ht[c] > 0.0f) || !(nu_wie[c] > 0.0f) || !std::isfinite(nu_ht[c]) || !std::isfinite(nu_wie[c]))
            return fail(B4D_ERR_INVALID, "relative variances must be positive and finite");
    std::memcpy(h->nu_ht, nu_ht, sizeof(h->nu_ht));
    std::memcpy(h->nu_wie, nu_wie, sizeof(h->nu_wie));
    h->psd = true;
    return 0;
}

int b4d_coherence_gate(b4d_handle *h, const float *raw, const uint64_t *labels, int64_t n, const int64_t shape[3],
                       double min_autocorr, double max_highfreq_frac, int64_t min_segment_voxels, double smooth_sigma,
                       int lag, uint8_t *reject, b4d_segment_score *seg, int64_t max_segments, int64_t *seg_count,
                       int in_on_device) {
    if (!h || !raw || !labels || !shape || !reject || n < 1) return fail(B4D_ERR_INVALID, "NULL argument or n < 1");
    for (int i = 0; i < 3; ++i)
        if (shape[i] < 1 || shape[i] > 65535) return fail(B4D_ERR_INVALID, "every dimension must be in [1, 65535]");
    if (!(smooth_sigma > 0) || smooth_sigma > 8.0) return fail(B4D_ERR_INVALID, "smooth_sigma must be in (0, 8]");
    if (lag < 1) return fail(B4D_ERR_INVALID, "lag must be >= 1");
    if (seg && (!seg_count || max_segments < 1)) return fail(B4D_ERR_INVALID, "seg needs seg_count and max_segments");
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int D = (int)shape[0], H = (int)shape[1], W = (int)shape[2];
    const long long V = (long long)D * H * W, TV = V * n;
    constexpr int CAP = 1024, NS = 23;
    // scipy.ndimage.gaussian_filter: radius int(truncate * sigma + 0.5), truncate = 4; weights exp(-x^2 / (2 sigma^2))
    // normalised to sum 1, float64
    const int radius = (int)(4.0 * smooth_sigma + 0.5);
    std::vector<double> w((size_t)2 * radius + 1);
    double wsum = 0.0;
    for (int k = -radius; k <= radius; ++k) wsum += (w[(size_t)(k + radius)] = std::exp(-0.5 / (smooth_sigma * smooth_sigma) * k * k));
    for (auto &v : w) v /= wsum;
    B4D_TRY(h->coh_x.ensure((size_t)TV * sizeof(double)));
    B4D_TRY(h->coh_sm.ensure((size_t)TV * sizeof(double)));
    B4D_TRY(h->coh_tmp.ensure((size_t)TV * sizeof(double)));
    B4D_TRY(h->coh_keys.ensure((size_t)n * CAP * sizeof(unsigned long long)));
    B4D_TRY(h->coh_sums.ensure((size_t)n * CAP * NS * sizeof(double) + 64));
    B4D_TRY(h->coh_w.ensure(w.size() * sizeof(double) + 64));
    const float *d_raw = raw;
    const unsigned long long *d_lab = reinterpret_cast<const unsigned long long *>(labels);
    if (!in_on_device) {
        B4D_TRY(h->in.ensure((size_t)TV * sizeof(float)));
        B4D_TRY(h->coh_lab.ensure((size_t)TV * sizeof(unsigned long long)));
        CU_TRY(copy_in(h, h->in.p, raw, (size_t)TV * sizeof(float), 0, s));
        CU_TRY(copy_in(h, h->coh_lab.p, labels, (size_t)TV * sizeof(unsigned long long), 0, s));
        d_raw = h->in.as<float>();
        d_lab = h->coh_lab.as<unsigned long long>();
    }
    CU_TRY(cudaMemcpyAsync(h->coh_w.p, w.data(), w.size() * sizeof(double), cudaMemcpyHostToDevice, s));
    int *d_over = reinterpret_cast<int *>(h->coh_w.as<char>() + w.size() * sizeof(double));
    b4d_launch_coherence(d_raw, d_lab, D, H, W, n, lag, radius, h->coh_w.as<double>(), h->coh_x.as<double>(),
                         h->coh_sm.as<double>(), h->coh_tmp.as<double>(), h->coh_keys.as<unsigned long long>(), CAP,
                         h->coh_sums.as<double>(), d_over, s);
    CU_TRY(cudaGetLastError());
    std::vector<unsigned long long> keys((size_t)n * CAP);
    std::vector<double> sums((size_t)n * CAP * NS);
    int over = 0;
    CU_TRY(cudaMemcpyAsync(keys.data(), h->coh_keys.p, keys.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaMemcpyAsync(sums.data(), h->coh_sums.p, sums.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaMemcpyAsync(&over, d_over, sizeof(int), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    if (over) return fail(B4D_ERR_UNSUPPORTED, "a patch holds more than 1024 distinct labels");
    for (int64_t i = 0; i < n; ++i) {
        reject[i] = 0;
        int64_t cnt = 0;
        for (int slot = 0; slot < CAP; ++slot) {
            const unsigned long long key = keys[(size_t)i * CAP + slot];
            if (!key) continue;
            const double *q = &sums[((size_t)i * CAP + slot) * NS];
            const double nv = q[0];
            // local_autocorr (metrics.py:96-112): per axis, pairs inside the segment; skipped when fewer than two
            // pairs or a standard deviation below 1e-6; mean over the axes left, 1.0 when none is
            double acs = 0.0;
            int nax = 0;
            for (int a = 0; a < 3; ++a) {
                const double *p = q + 5 + 6 * a;
                const double np_ = p[0];
                if (np_ < 2.0) continue;
                const double mx = p[1] / np_, my = p[2] / np_;
                const double vx = std::max(p[3] / np_ - mx * mx, 0.0), vy = std::max(p[4] / np_ - my * my, 0.0);
                if (std::sqrt(vx) < 1e-6 || std::sqrt(vy) < 1e-6) continue;
                acs += (p[5] / np_ - mx * my) / std::sqrt(vx * vy);
                ++nax;
            }
            const double autocorr = nax ? acs / nax : 1.0;
            // highfreq_energy_fraction (metrics.py:148-155): population variances over the segment
            const double mv = q[1] / nv, mh = q[3] / nv;
            const double vv = std::max(q[2] / nv - mv * mv, 0.0), vh = std::max(q[4] / nv - mh * mh, 0.0);
            const double hf = vv < 1e-12 ? 0.0 : vh / vv;
            if ((int64_t)nv >= min_segment_voxels && autocorr < min_autocorr && hf > max_highfreq_frac) reject[i] = 1;
            if (seg && cnt < max_segments) {
                b4d_segment_score &o = seg[i * max_segments + cnt];
                o.label = key;
                o.voxels = (int64_t)nv;
                o.autocorr = autocorr;
                o.highfreq = hf;
            }
            ++cnt;
        }
        if (seg_count) seg_count[i] = cnt;
    }
    return 0;
}

int b4d_debug_accumulators(b4d_handle *h, int64_t *numq, int64_t *wmap, int64_t n) {
    if (!h || !numq || !wmap || n < 1) return fail(B4D_ERR_INVALID, "NULL argument");
    CU_TRY(cudaSetDevice(h->device));
    if (h->numq.cap < (size_t)n * sizeof(long long) || h->gmap.cap < (size_t)n * sizeof(uint32_t))
        return fail(B4D_ERR_INVALID, "no accumulators of that size");
    CU_TRY(cudaStreamSynchronize(h->stream));
    CU_TRY(cudaMemcpy(numq, h->numq.p, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost));
    std::vector<uint32_t> g((size_t)n);
    CU_TRY(cudaMemcpy(g.data(), h->gmap.p, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < n; ++i) wmap[i] = (int64_t)g[(size_t)i];
    return 0;
}

int b4d_measure_pipe_peaks(b4d_handle *h, double out[4]) {
    if (!h || !out) return fail(B4D_ERR_INVALID, "NULL argument");
    CU_TRY(cudaSetDevice(h->device));
    B4D_TRY(h->sink.ensure(64));
    cudaStream_t s = h->stream;
    cudaEvent_t a, b;
    CU_TRY(cudaEventCreate(&a));
    CU_TRY(cudaEventCreate(&b));
    for (int which = 0; which < 4; ++which) {
        double best = 0.0;
        for (int rep = 0; rep < 4; ++rep) {
            const int iters = rep == 0 ? 64 : 2048;
            cudaEventRecord(a, s);
            const double ops = b4d_launch_pipe_bench(which, iters, h->sink.as<unsigned>(), s);
            cudaEventRecord(b, s);
            CU_TRY(cudaEventSynchronize(b));
            float ms = 0.f;
            cudaEventElapsedTime(&ms, a, b);
            if (rep > 0 && ms > 0.f) best = std::max(best, ops / (ms * 1e-3));
        }
        out[which] = best;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    CU_TRY(cudaGetLastError());
    return 0;
}

}  // extern "C"
