// b4d_match.cu — K0 (block energies), tile classification and K1 / K4 (exact-integer block matching)
// on a uint16 image.
//
// Contract (DESIGN.md §3.2, SURVEY Appendix A): for every reference block
// (4x4x4, origins on the step-3 grid plus the flush origin N-4) compute the
// exact SSD to every candidate origin of the Ns^3 window clipped to the volume,
// accept SSD <= tau, order by (SSD, window index), keep the first
// K' = 2^floor(log2(min(K, accepted))).
//
// Arithmetic.  SSD(a, b) = S2(a) + S2(b) - 2 * sum(a*b), with S2 the block energy sum(v^2), all exact.
// K0 writes {S2 mod 2^32, S1 | (S2 >> 32) << 24} for every block origin once per stage (S1 = block sum).
// The cross term never uses one multiply per voxel pair:
//   * byte tiles (the staged neighbourhood spans <= 255 counts): v - tile_min fits a byte, four products per
//     IDP.4A (dp4a), energies of the centred bytes rebuilt in shared memory; k_match<.., BYTE = true>;
//   * all other tiles: the REFERENCE block is split into byte planes of r - r_min (one plane when the block spans
//     <= 255 counts, else two), candidates stay 16-bit, two products per IDP.2A (dp2a);
//     sum(a r) = sum(a rl) + 256 sum(a rh) + r_min S1(a).  On a narrow tile (range <= 8191, every SSD < 2^32) the
//     combination runs modulo 2^32, on a wide tile exactly in 64 bits; k_match<.., BYTE = false>.
// Tiles are classified beforehand by the exact range of their neighbourhood (k_plane_ranges, k_tile_class); each
// instantiation exits at once on a tile of the other class.
//
// Mapping.  One CTA per 4x4x4 tile of reference blocks; the (Ns+12)^3 voxel neighbourhood and the (Ns+9)^3 table
// entries are staged once in shared memory (TMA box loads: the uint16 window of byte tiles, the 8-byte table of the
// other tiles; cp.async for the rest and for volumes whose row pitch breaks the 16-byte rule) and serve all 64
// reference blocks.  One warp per reference block — in the byte kernel per PAIR of blocks that are neighbours in x,
// which search the same rows.  A lane owns one (dz, dy) row of the window at a time and slides along dx with Ns
// accumulators (per reference) in registers.  Shared-memory strides are padded so that the 32 rows a warp reads at
// once fall in 32 distinct banks (bank = B * (Ns*dz + dy) mod 32 with B odd).
//
// Selection is exact and deterministic: key = SSD << KB | window index (unique),
// rejected candidates get 0xFFFFFFFF.  Rows are visited centre-out so the good
// matches arrive first; a running per-lane minimum (second minimum for K = 32)
// gives, through one 32-lane bitonic sort, an upper bound B with at least K keys
// <= B; only keys <= B are appended to a small per-warp survivor list, which is
// rank-sorted at the end.  If the list overflows (adversarial key order) the warp
// retries once with the final bound, then falls back to K rounds of "smallest key greater than the previous one".
#include <algorithm>
#include <cstring>
#include <type_traits>

#include "b4d_common.cuh"
#include "b4d_tma.cuh"

namespace {

constexpr int WARPS = 8;
constexpr int CAP = 512;  // survivor list entries per warp

// ---- shared-memory geometry (all constexpr in NS) ---------------------------
template <int NS>
struct Geo {
    static constexpr int R = NS / 2;
    static constexpr int E = NS + 12;   // staged voxels per axis
    static constexpr int EC = NS + 9;   // staged block origins per axis (E - 3)
    static constexpr int UNITS = NS * NS;
    static constexpr int ITERS = (UNITS + 31) / 32;
    static constexpr int KB = (NS * NS * NS <= 2048) ? 11 : 12;
    // uint16 window: row stride 2*BW elements (BW odd words), plane stride 2*AW
    static constexpr int BW = ((E + 1) / 2) | 1;
    static constexpr int AW0 = E * BW;
    static constexpr int AW = AW0 + (((NS * BW) % 32 - AW0 % 32) + 32) % 32;
    static constexpr int SY = 2 * BW, SZ = 2 * AW;
    static constexpr int WIN_ELEMS = E * SZ;
    // uint32 energies: row stride BC (odd words), plane stride AC
    static constexpr int BC = EC | 1;
    static constexpr int AC0 = EC * BC;
    static constexpr int AC = AC0 + (((NS * BC) % 32 - AC0 % 32) + 32) % 32;
    static constexpr int S2_WORDS = EC * AC;
    // general kernel: the {S2, S1} table is DENSE ([EC][EC][TBW] entries of 8 bytes), the layout a TMA box load
    // produces; TBW = EC + 2 leaves room for the 16-byte alignment of the box origin (one entry)
    static constexpr int TBW = EC + 2;
    static constexpr int TAC = EC * TBW;
    static constexpr uint32_t TAB_BOX_BYTES = (uint32_t)TBW * EC * EC * 8;
    static constexpr size_t WIN_BYTES = (((size_t)WIN_ELEMS * 2 + 127) & ~(size_t)127);
    static constexpr size_t SMEM = WIN_BYTES + (size_t)TAB_BOX_BYTES;
    // byte window: row stride RSW words (odd), plane stride PSW = NS*RSW (mod 32): the 32
    // (dz, dy) rows a warp reads at once fall in 32 distinct banks
    static constexpr int RW = (E + 3) / 4;     // words of a row that hold data
    static constexpr int RSW = (RW + 1) | 1;   // > RW: the realignment reads one word past
    static constexpr int PSW0 = E * RSW;
    static constexpr int PSW = PSW0 + (((NS * RSW) % 32 - PSW0 % 32) + 32) % 32;
    static constexpr int BWIN_WORDS = E * PSW;
    static constexpr int NWR = (NS + 9) / 4;   // row words a lane loads: bytes [a, a + NS + 3), a <= 3
    // byte kernel: byte window + the S2' table, whose space first holds the raw uint16 window
    static constexpr size_t TAB_B0 =
        (size_t)S2_WORDS * 4 > (size_t)WIN_ELEMS * 2 ? (size_t)S2_WORDS * 4 : (size_t)WIN_ELEMS * 2;
    // TMA staging of the byte kernel: one 4-D box (BOXW x E x E x 1 uint16) lands DENSE in the table space; the byte
    // conversion reads it from there.  Measured on B200 (tools/tma_check.cu): the innermost start coordinate has to be
    // a multiple of 16 bytes (8 voxels) — an unaligned one raises "illegal instruction" — so the box starts at the
    // aligned column below the window and is up to 7 columns wider, rounded to the 16-byte rule; 128-byte aligned
    // destination; the barrier initialisation needs fence.proxy.async before the TMA unit may use it.
    static constexpr int BOXW = (4 * RW + 7 + 7) & ~7;  // the conversion reads whole words of 4 voxels from column xb <= 7 on
    static constexpr uint32_t BOX_BYTES = (uint32_t)BOXW * E * E * 2;
    static constexpr size_t TAB_B = TAB_B0 > (size_t)BOX_BYTES ? TAB_B0 : (size_t)BOX_BYTES;
    static constexpr size_t BWIN_BYTES = (((size_t)BWIN_WORDS * 4 + 127) & ~(size_t)127);
    static constexpr size_t SMEM_B = BWIN_BYTES + TAB_B;
    // centre-out visiting order of the 32-unit groups: mc, mc+1, mc-1, mc+2, ...
    // packed 4 bits per entry so the device reads it with a shift and a mask
    static constexpr int order_at(int it) {
        const int mc = (UNITS / 2) / 32;
        int count = 0;
        for (int k = 0; k < 2 * ITERS + 2; ++k) {
            const int off = (k + 1) / 2;
            const int m = (k & 1) ? mc + off : mc - off;
            if (m < 0 || m >= ITERS) continue;
            if (count == it) return m;
            ++count;
        }
        return 0;
    }
    static constexpr unsigned long long order_pack() {
        unsigned long long v = 0;
        for (int it = 0; it < ITERS; ++it) v |= (unsigned long long)order_at(it) << (4 * it);
        return v;
    }
    static constexpr unsigned long long ORDER = order_pack();
};

// ------------------------------------------------------------------ K0 ------
// For every block origin (z,y,x) with z <= D-4, y <= H-4, x <= W-4 (others are left
// untouched): S2 = sum over the 4x4x4 block of u^2 (exact, < 2^38) and S1 = sum of u
// (< 2^22), packed as uint2 {S2 mod 2^32, S1 | (S2 >> 32) << 24}.
// Separable box sums without shared memory or barriers: a WARP owns K0_TY x 29 (y, x) origins and marches along
// z.  Lane i holds column x0 + i of the K0_TY + 3 rows of a plane (the next plane's loads are issued before the
// current one is summed); the 4-tap sum along x takes the three right-hand neighbours by shuffle (lanes 29-31
// only feed them), the sums along y and z are register arithmetic (pair sums, three older plane sums per row).
// HBM-bound: 2 B read + 8 B written per voxel.
constexpr int K0_TY = 8, K0_TX = 29, K0_ZC = 128, K0_WARPS = 8;
__global__ void __launch_bounds__(K0_WARPS * 32) k_block_energy(const uint16_t *__restrict__ u, uint2 *__restrict__ s21,
                                                               int D, int H, int W, int nvol, int zo0, int zo1) {
    const int lane = threadIdx.x & 31;
    const int ntx = (W - 3 + K0_TX - 1) / K0_TX, nty = (H - 3 + K0_TY - 1) / K0_TY;
    const int nzc = (zo1 - zo0 + K0_ZC - 1) / K0_ZC;  // origins z in [zo0, zo1) only
    long long t = (long long)blockIdx.x * K0_WARPS + (threadIdx.x >> 5);
    if (t >= (long long)ntx * nty * nzc * nvol) return;  // warp-uniform
    const int txi = (int)(t % ntx);
    t /= ntx;
    const int tyi = (int)(t % nty);
    t /= nty;
    const int zci = (int)(t % nzc);
    const int vol = (int)(t / nzc);
    const int x0 = txi * K0_TX, y0 = tyi * K0_TY, z0 = zo0 + zci * K0_ZC, z1 = min(z0 + K0_ZC, zo1);
    const uint16_t *__restrict__ uv = u + (long long)vol * D * H * W;
    uint2 *__restrict__ ov = s21 + (long long)vol * D * H * W;
    const int gx = x0 + lane;
    const bool cin = gx < W;
    const bool wx = lane < K0_TX && gx <= W - 4;
    const long long plane = (long long)H * W;
    const uint16_t *col = uv + (cin ? gx : 0);

    uint32_t nxt[K0_TY + 3];
    auto load_plane = [&](int z) {
        const uint16_t *pz = col + (long long)z * plane;
#pragma unroll
        for (int r = 0; r < K0_TY + 3; ++r) {
            const int gy = y0 + r;
            nxt[r] = (cin && gy < H) ? (uint32_t)__ldg(pz + (long long)gy * W) : 0u;
        }
    };
    unsigned long long q1[K0_TY], q2[K0_TY], q3[K0_TY];  // plane sums of z-1, z-2, z-3 per output row
    uint32_t l1[K0_TY], l2[K0_TY], l3[K0_TY];
#pragma unroll
    for (int r = 0; r < K0_TY; ++r) {
        q1[r] = q2[r] = q3[r] = 0ull;
        l1[r] = l2[r] = l3[r] = 0u;
    }
    load_plane(z0);
    for (int z = z0; z < z1 + 3; ++z) {  // z1 + 2 <= D - 1
        uint32_t cur[K0_TY + 3];
#pragma unroll
        for (int r = 0; r < K0_TY + 3; ++r) cur[r] = nxt[r];
        if (z + 1 < z1 + 3) load_plane(z + 1);
        // sums along x: this lane's value and its three right-hand neighbours
        unsigned long long x2[K0_TY + 3];
        uint32_t x1[K0_TY + 3];
#pragma unroll
        for (int r = 0; r < K0_TY + 3; ++r) {
            const uint32_t a = cur[r];
            const uint32_t b = __shfl_down_sync(B4D_FULL, a, 1), c = __shfl_down_sync(B4D_FULL, a, 2),
                           d = __shfl_down_sync(B4D_FULL, a, 3);
            x1[r] = a + b + c + d;
            x2[r] = (unsigned long long)(a * a) + (b * b) + (unsigned long long)(c * c) + (d * d);
        }
        // sums along y through pair sums, then the sliding sum along z
        unsigned long long p2[K0_TY + 2];
        uint32_t p1[K0_TY + 2];
#pragma unroll
        for (int r = 0; r < K0_TY + 2; ++r) {
            p2[r] = x2[r] + x2[r + 1];
            p1[r] = x1[r] + x1[r + 1];
        }
        const bool out_z = z >= z0 + 3;
        uint2 *orow = ov + (long long)(z - 3) * plane + gx;
#pragma unroll
        for (int r = 0; r < K0_TY; ++r) {
            const unsigned long long q0 = p2[r] + p2[r + 2];
            const uint32_t l0 = p1[r] + p1[r + 2];
            if (out_z && wx && y0 + r <= H - 4) {
                const unsigned long long sq = (q0 + q1[r]) + (q2[r] + q3[r]);
                const uint32_t m = (l0 + l1[r]) + (l2[r] + l3[r]);
                // .x = S2 mod 2^32; .y = S1 | (S2 >> 32) << 24
                orow[(long long)(y0 + r) * W] = make_uint2((uint32_t)sq, m | ((uint32_t)(sq >> 32) << 24));
            }
            q3[r] = q2[r];
            q2[r] = q1[r];
            q1[r] = q0;
            l3[r] = l2[r];
            l2[r] = l1[r];
            l1[r] = l0;
        }
    }
}

// The same sums with the input planes brought in by TMA (the production path when W % 8 == 0): a CTA of 4 warps owns
// K0_TY x 112 origins and marches along z; one 4-D box load per plane (120 x 11 uint16, zero fill outside the
// volume) lands in a ring of K0T_NST shared-memory stages, so that 8 planes (21 KB) per CTA are in flight without a
// register or an LSU slot being spent on them.  Full / empty mbarriers per stage; thread 0 refills the stage of
// plane i - 1 after its own work on plane i (the other warps have normally released it by then).  Each warp reads
// its 28 + 3 columns from the stage (one 2-byte LDS per row) and works on packed 64-bit words
// v^2 | v << 40: every partial sum of S2 stays below 2^38 and of S1 below 2^22, so one 64-bit addition serves both.
// Rows are summed first (registers), then columns by two shuffles (v + right neighbour, pair + pair two lanes on);
// the three older plane sums per row are kept by phase (z mod 3), nothing is moved.
constexpr int K0T_WARPS = 2, K0T_WX = 28, K0T_TX = K0T_WARPS * K0T_WX, K0T_BOXW = 64, K0T_ROWS = K0_TY + 3, K0T_NST = 8;
constexpr uint32_t K0T_BOX_BYTES = K0T_BOXW * K0T_ROWS * 2;
constexpr int K0T_STAGE = ((int)K0T_BOX_BYTES + 127) / 128 * 128;
static_assert(K0T_TX % 8 == 0 && K0T_BOXW % 8 == 0 && K0T_BOXW >= K0T_TX + 3 && K0T_BOXW >= (K0T_WARPS - 1) * K0T_WX + 32,
              "TMA box of K0");
__global__ void __launch_bounds__(K0T_WARPS * 32) k_block_energy_tma(const __grid_constant__ CUtensorMap tmap,
                                                                    uint2 *__restrict__ s21, int D, int H, int W, int nvol,
                                                                    int zo0, int zo1) {
    __shared__ __align__(128) unsigned char s_buf[K0T_NST * K0T_STAGE];
    __shared__ __align__(8) unsigned long long s_full[K0T_NST], s_empty[K0T_NST];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ntx = (W - 3 + K0T_TX - 1) / K0T_TX, nty = (H - 3 + K0_TY - 1) / K0_TY;
    const int nzc = (zo1 - zo0 + K0_ZC - 1) / K0_ZC;
    long long t = blockIdx.x;
    const int txi = (int)(t % ntx);
    t /= ntx;
    const int tyi = (int)(t % nty);
    t /= nty;
    const int zci = (int)(t % nzc);
    const int vol = (int)(t / nzc);
    const int x0 = txi * K0T_TX, y0 = tyi * K0_TY, z0 = zo0 + zci * K0_ZC, z1 = min(z0 + K0_ZC, zo1);
    const int nplanes = z1 + 3 - z0;  // input planes z0 .. z1 + 2 (<= D - 1)
    const uint32_t buf0 = (uint32_t)__cvta_generic_to_shared(s_buf);
    const uint32_t full0 = (uint32_t)__cvta_generic_to_shared(s_full), empty0 = (uint32_t)__cvta_generic_to_shared(s_empty);
    if (threadIdx.x == 0) {
        for (int i = 0; i < K0T_NST; ++i) {
            mbar_init(full0 + 8u * i, 1);
            mbar_init(empty0 + 8u * i, K0T_WARPS);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 0; i < min(K0T_NST, nplanes); ++i) {
            mbar_expect_tx(full0 + 8u * i, K0T_BOX_BYTES);
            tma_load_4d(buf0 + (uint32_t)(i * K0T_STAGE), &tmap, full0 + 8u * i, x0, y0, z0 + i, vol);
        }
    }
    const int gx = x0 + warp * K0T_WX + lane;
    const bool wx = lane < K0T_WX && gx <= W - 4;
    const long long plane = (long long)H * W;
    uint2 *ocol = s21 + (long long)vol * D * plane + gx;
    unsigned long long h[3][K0_TY];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int r = 0; r < K0_TY; ++r) h[k][r] = 0ull;

    auto step = [&](auto PH, int i) {
        constexpr int ph = decltype(PH)::value;
        const int slot = i % K0T_NST;
        mbar_wait(full0 + 8u * slot, (uint32_t)((i / K0T_NST) & 1));
        const uint16_t *sp = reinterpret_cast<const uint16_t *>(s_buf + slot * K0T_STAGE) + warp * K0T_WX + lane;
        uint32_t a[K0T_ROWS];
#pragma unroll
        for (int r = 0; r < K0T_ROWS; ++r) a[r] = sp[r * K0T_BOXW];
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8u * slot);
        if (threadIdx.x == 0 && i >= 1 && i - 1 + K0T_NST < nplanes) {  // refill the stage of the previous plane
            const int ps = (i - 1) % K0T_NST;
            mbar_wait(empty0 + 8u * ps, (uint32_t)(((i - 1) / K0T_NST) & 1));
            mbar_expect_tx(full0 + 8u * ps, K0T_BOX_BYTES);
            tma_load_4d(buf0 + (uint32_t)(ps * K0T_STAGE), &tmap, full0 + 8u * ps, x0, y0, z0 + i - 1 + K0T_NST, vol);
        }
        unsigned long long w[K0T_ROWS], pr[K0T_ROWS - 1];
#pragma unroll
        for (int r = 0; r < K0T_ROWS; ++r) w[r] = (unsigned long long)(a[r] * a[r]) | ((unsigned long long)a[r] << 40);
#pragma unroll
        for (int r = 0; r < K0T_ROWS - 1; ++r) pr[r] = w[r] + w[r + 1];
        const bool out_z = i >= 3;
        uint2 *orow = ocol + (long long)(z0 + i - 3) * plane;
#pragma unroll
        for (int r = 0; r < K0_TY; ++r) {
            const unsigned long long c = pr[r] + pr[r + 2];                           // 4 rows of this column
            const unsigned long long c2 = c + __shfl_down_sync(B4D_FULL, c, 1);      // columns x, x + 1
            const unsigned long long q0 = c2 + __shfl_down_sync(B4D_FULL, c2, 2);    // columns x .. x + 3
            if (out_z && wx && y0 + r <= H - 4) {
                const unsigned long long sq = (q0 + h[0][r]) + (h[1][r] + h[2][r]);
                const uint32_t hi = (uint32_t)(sq >> 32);  // bits 0-5: S2 >> 32, bits 8-29: S1
                // .x = S2 mod 2^32; .y = S1 | (S2 >> 32) << 24 = hi rotated right by 8
                orow[(long long)(y0 + r) * W] = make_uint2((uint32_t)sq, __funnelshift_r(hi, hi, 8));
            }
            h[ph][r] = q0;  // replaces the sum of plane i - 3
        }
    };
    for (int i = 0; i < nplanes; i += 3) {
        step(std::integral_constant<int, 0>{}, i);
        if (i + 1 < nplanes) step(std::integral_constant<int, 1>{}, i + 1);
        if (i + 2 < nplanes) step(std::integral_constant<int, 2>{}, i + 2);
    }
}

// ------------------------------------------------- tile classification ------
// EXACT range of every matcher tile's staged neighbourhood [b, b + E)^3 (clipped to the volume), separably:
// k_plane_ranges: per voxel plane z and tile (ty, tx), min | max << 16 over the (y, x) window of that tile;
// k_tile_class: per tile, the reduction of those over its z window.  (Round 1 took the range over the aligned 4^3
// cells covering the neighbourhood — up to 5 voxels wider per axis, which pushed 12 % of the tiles of the benchmark
// volume from the byte kernel to the general one.)
// One CTA per (plane, ty): column min / max over the <= E rows of the window go to shared memory, segment by
// segment of 64 tiles along x; one warp per tile then reduces its <= E columns.
template <int NS>
__global__ void __launch_bounds__(256) k_plane_ranges(const uint16_t *__restrict__ u, const B4dGeom g,
                                                      uint32_t *__restrict__ rxy, int z0, int z1) {
    using G = Geo<NS>;
    constexpr int SEG_T = 64, SEG_W = 12 * (SEG_T - 1) + G::E;  // columns spanned by 64 consecutive tiles
    __shared__ uint32_t s_col[SEG_W];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long t = blockIdx.x;
    const int tyi = (int)(t % g.ty);
    t /= g.ty;
    const int z = z0 + (int)(t % (z1 - z0));
    const int vol = (int)(t / (z1 - z0));
    const int by = g.refy[tyi * 4] - G::R;
    const int ya = max(by, 0), yb = min(by + G::E, g.H);
    const uint16_t *pl = u + (long long)vol * g.vol_stride + (long long)z * g.H * g.W;
    uint32_t *out = rxy + (((long long)vol * g.D + z) * g.ty + tyi) * g.tx;
    const bool vec4 = (g.W & 3) == 0 && (reinterpret_cast<uintptr_t>(u) & 7) == 0;
    for (int ts = 0; ts < g.tx; ts += SEG_T) {
        const int te = min(ts + SEG_T, g.tx);
        const int xs = g.refx[ts * 4] - G::R;                       // first column of the segment (may be < 0)
        const int xe = min(g.refx[(te - 1) * 4] - G::R + G::E, g.W);  // one past its last column
        __syncthreads();
        if (vec4) {
            // four columns per thread and load (8 bytes): the pass is bound by the number of load instructions
            const int x_first = max(xs, 0);
            for (int x4 = (x_first & ~3) + 4 * (int)threadIdx.x; x4 < xe; x4 += 4 * 256) {
                uint32_t mn[4] = {0xFFFFu, 0xFFFFu, 0xFFFFu, 0xFFFFu}, mx[4] = {0u, 0u, 0u, 0u};
                for (int y = ya; y < yb; ++y) {
                    const uint2 v = __ldg(reinterpret_cast<const uint2 *>(pl + (long long)y * g.W + x4));
                    const uint32_t q[4] = {v.x & 0xFFFFu, v.x >> 16, v.y & 0xFFFFu, v.y >> 16};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        mn[k] = min(mn[k], q[k]);
                        mx[k] = max(mx[k], q[k]);
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int x = x4 + k;
                    if (x >= x_first && x < xe) s_col[x - xs] = mn[k] | (mx[k] << 16);
                }
            }
        } else {
            for (int x = max(xs, 0) + threadIdx.x; x < xe; x += 256) {
                uint32_t mn = 0xFFFFu, mx = 0u;
                for (int y = ya; y < yb; ++y) {
                    const uint32_t q = __ldg(pl + (long long)y * g.W + x);
                    mn = min(mn, q);
                    mx = max(mx, q);
                }
                s_col[x - xs] = mn | (mx << 16);
            }
        }
        __syncthreads();
        for (int ti = ts + warp; ti < te; ti += 8) {
            const int bx = g.refx[ti * 4] - G::R;
            const int x = bx + lane;
            uint32_t mn = 0xFFFFu, mx = 0u;
            if (lane < G::E && x >= 0 && x < g.W) {
                const uint32_t c = s_col[x - xs];
                mn = c & 0xFFFFu;
                mx = c >> 16;
            }
            mn = __reduce_min_sync(B4D_FULL, mn);
            mx = __reduce_max_sync(B4D_FULL, mx);
            if (lane == 0) out[ti] = mn | (mx << 16);
        }
    }
}
// One warp per matcher tile.  tcls[tile]: bit 16 = the range fits a byte (then bits 0-15 hold the minimum),
// bit 17 = "narrow", range <= 8191 (every SSD < 2^32).
template <int NS>
__global__ void __launch_bounds__(256) k_tile_class(const uint32_t *__restrict__ rxy, const B4dGeom g,
                                                    uint32_t *__restrict__ tcls, long long tile0, long long tile1) {
    using G = Geo<NS>;
    static_assert(G::E <= 32, "one lane per plane of the z window");
    const int lane = threadIdx.x & 31;
    const long long tile = tile0 + (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (tile >= tile1) return;
    long long t = tile;
    const int tx = (int)(t % g.tx);
    t /= g.tx;
    const int ty = (int)(t % g.ty);
    t /= g.ty;
    const int tz = (int)(t % g.tz);
    const int vol = (int)(t / g.tz);
    const int bz = g.refz[tz * 4] - G::R;
    const int z = bz + lane;
    uint32_t mn = 0xFFFFu, mx = 0u;
    if (lane < G::E && z >= 0 && z < g.D) {
        const uint32_t c = __ldg(rxy + (((long long)vol * g.D + z) * g.ty + ty) * g.tx + tx);
        mn = c & 0xFFFFu;
        mx = c >> 16;
    }
    mn = __reduce_min_sync(B4D_FULL, mn);
    mx = __reduce_max_sync(B4D_FULL, mx);
    if (lane == 0) {
        const uint32_t range = mx >= mn ? mx - mn : 0u;
        // bit 18: the four reference columns of the tile exist and sit 3 voxels apart (no flush origin among them):
        // the byte kernel then matches them as two pairs
        const int ix0 = tx * 4;
        const uint32_t reg = (ix0 + 3 < g.nrx && g.refx[ix0 + 3] - g.refx[ix0] == 9) ? (1u << 18) : 0u;
        tcls[tile] = (range <= 255u ? ((3u << 16) | mn) : (range <= 8191u ? (2u << 16) : 0u)) | reg;
    }
}

// ------------------------------------------------------------ helpers -------
// key = SSD * 2^KB + window index as ONE multiply-add (IMAD pipe) instead of a shift and an OR (ALU pipe, which is the
// busier one in these kernels); the low KB bits of the product are zero, so the sum equals the OR
__device__ __forceinline__ uint32_t mad_key(uint32_t ssd, uint32_t scale, uint32_t idx) {
    uint32_t k;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(k) : "r"(ssd), "r"(scale), "r"(idx));
    return k;
}
__device__ __forceinline__ uint32_t warp_min_u32(uint32_t v) { return __reduce_min_sync(B4D_FULL, v); }

// K-th smallest (0-based index kth) of one value per lane: 32-lane bitonic sort.
__device__ __forceinline__ uint32_t kth_smallest32(uint32_t v, int kth, int lane) {
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const uint32_t o = __shfl_xor_sync(B4D_FULL, v, j);
            const bool up = (lane & k) == 0;  // ascending half (k == 32: all ascending)
            const bool lower = (lane & j) == 0;
            const uint32_t mn = min(v, o), mx = max(v, o);
            v = (lower == up) ? mn : mx;
        }
    }
    return __shfl_sync(B4D_FULL, v, kth);
}

// Byte path: cross terms of one (dz, dy) row of candidates from the byte window.
// `base` points at the aligned word that holds byte wx0 of the first row, `sel` is the
// PRMT selector of the run-time alignment wx0 & 3, refw[16] the reference block rows.
template <int NS>
__device__ __forceinline__ void bcorr_row(const uint32_t *__restrict__ base, uint32_t sel, const uint32_t (&refw)[16],
                                          uint32_t (&acc)[NS]) {
    using G = Geo<NS>;
#pragma unroll
    for (int j = 0; j < NS; ++j) acc[j] = 0u;
#pragma unroll
    for (int z = 0; z < 4; ++z) {
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            uint32_t w[G::NWR], q[G::NWR - 1];
#pragma unroll
            for (int i = 0; i < G::NWR; ++i) w[i] = base[z * G::PSW + y * G::RSW + i];
#pragma unroll
            for (int i = 0; i < G::NWR - 1; ++i) q[i] = __byte_perm(w[i], w[i + 1], sel);  // bytes wx0 + 4i ..
            const uint32_t r = refw[z * 4 + y];
#pragma unroll
            for (int j = 0; j < NS; ++j) {
                const uint32_t c = (j & 3) == 0   ? q[j >> 2]
                                   : (j & 3) == 1 ? __byte_perm(q[j >> 2], q[(j >> 2) + 1], 0x4321)
                                   : (j & 3) == 2 ? __byte_perm(q[j >> 2], q[(j >> 2) + 1], 0x5432)
                                                  : __byte_perm(q[j >> 2], q[(j >> 2) + 1], 0x6543);
                acc[j] = __dp4a(c, r, acc[j]);
            }
        }
    }
}

// The same for TWO reference blocks that are neighbours in x (origins 3 voxels apart): their windows cover the same
// (dz, dy) rows, so one set of row loads and realignments feeds both.  Candidate j of A sits at byte wx0 + j, candidate
// j of B at byte wx0 + 3 + j: NS + 3 extracted words instead of 2 NS, NQ + 1 loads instead of 2 NWR.
template <int NS>
__device__ __forceinline__ void bcorr_row_pair(const uint32_t *__restrict__ base, uint32_t sel, const uint32_t (&refa)[16],
                                               const uint32_t (&refb)[16], uint32_t (&acca)[NS], uint32_t (&accb)[NS]) {
    using G = Geo<NS>;
    constexpr int NQ = (NS + 9) / 4;  // aligned words that cover bytes [0, NS + 6)
#pragma unroll
    for (int j = 0; j < NS; ++j) acca[j] = accb[j] = 0u;
#pragma unroll
    for (int z = 0; z < 4; ++z) {
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            uint32_t w[NQ + 1], q[NQ];
#pragma unroll
            for (int i = 0; i < NQ + 1; ++i) w[i] = base[z * G::PSW + y * G::RSW + i];
#pragma unroll
            for (int i = 0; i < NQ; ++i) q[i] = __byte_perm(w[i], w[i + 1], sel);  // bytes wx0 + 4i ..
            const uint32_t ra = refa[z * 4 + y], rb = refb[z * 4 + y];
            uint32_t c[NS + 3];
#pragma unroll
            for (int pp = 0; pp < NS + 3; ++pp)
                c[pp] = (pp & 3) == 0   ? q[pp >> 2]
                        : (pp & 3) == 1 ? __byte_perm(q[pp >> 2], q[(pp >> 2) + 1], 0x4321)
                        : (pp & 3) == 2 ? __byte_perm(q[pp >> 2], q[(pp >> 2) + 1], 0x5432)
                                        : __byte_perm(q[pp >> 2], q[(pp >> 2) + 1], 0x6543);
#pragma unroll
            for (int j = 0; j < NS; ++j) {
                acca[j] = __dp4a(c[j], ra, acca[j]);
                accb[j] = __dp4a(c[j + 3], rb, accb[j]);
            }
        }
    }
}

// Reference-byte path: sum(a * r') of one (dz, dy) row of candidates; a = uint16 window,
// r' = reference bytes (rw[16], one word per block row).  `base` = aligned word that holds
// window element wx0 - P of the first row, P = wx0 & 1; `sel` = PRMT selector that realigns
// two neighbouring words by P elements (0x3210 or 0x5432).
template <int NS>
__device__ __forceinline__ void r8corr_row(const uint32_t *__restrict__ base, uint32_t sel, const uint32_t (&rw)[16],
                                           uint32_t (&acc)[NS]) {
    using G = Geo<NS>;
    constexpr int NA = (NS + 4) / 2;  // pair words (v[2i], v[2i+1]) covering elements [0, NS + 3)
#pragma unroll
    for (int j = 0; j < NS; ++j) acc[j] = 0u;
#pragma unroll
    for (int z = 0; z < 4; ++z) {
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            uint32_t w[NA + 1], al[NA];
#pragma unroll
            for (int i = 0; i < NA + 1; ++i) w[i] = base[z * G::AW + y * G::BW + i];
#pragma unroll
            for (int i = 0; i < NA; ++i) al[i] = __byte_perm(w[i], w[i + 1], sel);
            const uint32_t r = rw[z * 4 + y];
#pragma unroll
            for (int j = 0; j < NS; ++j) {
                // pair words (v[j], v[j+1]) and (v[j+2], v[j+3])
                const uint32_t p0 = (j & 1) == 0 ? al[j / 2] : __byte_perm(al[j / 2], al[j / 2 + 1], 0x5432);
                const uint32_t p1 = (j & 1) == 0 ? al[j / 2 + 1] : __byte_perm(al[j / 2 + 1], al[j / 2 + 2], 0x5432);
                acc[j] = __dp2a_lo(p0, r, acc[j]);
                acc[j] = __dp2a_hi(p1, r, acc[j]);
            }
        }
    }
}

// cp.async with zero fill: copies `n` (0 or the full size) bytes, zero-fills the rest
__device__ __forceinline__ void cp_async4_zfill(uint32_t saddr, const void *g, uint32_t n) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(saddr), "l"(g), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async8_zfill(uint32_t saddr, const void *g, uint32_t n) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(saddr), "l"(g), "r"(n) : "memory");
}

// The same sums for the HIGH byte plane of a reference block that spans more than 255 counts
// (rare): rolled over the 16 block rows, reference bytes from shared memory, so that it adds
// one row body of code instead of sixteen.
template <int NS>
__device__ __forceinline__ void r8corr_row_rolled(const uint32_t *__restrict__ base, uint32_t sel,
                                                  const uint32_t *__restrict__ rw, uint32_t (&acc)[NS]) {
    using G = Geo<NS>;
    constexpr int NA = (NS + 4) / 2;
#pragma unroll
    for (int j = 0; j < NS; ++j) acc[j] = 0u;
#pragma unroll 1
    for (int row = 0; row < 16; ++row) {
        const uint32_t *b = base + (row >> 2) * G::AW + (row & 3) * G::BW;
        uint32_t w[NA + 1], al[NA];
#pragma unroll
        for (int i = 0; i < NA + 1; ++i) w[i] = b[i];
#pragma unroll
        for (int i = 0; i < NA; ++i) al[i] = __byte_perm(w[i], w[i + 1], sel);
        const uint32_t r = rw[row];
#pragma unroll
        for (int j = 0; j < NS; ++j) {
            const uint32_t p0 = (j & 1) == 0 ? al[j / 2] : __byte_perm(al[j / 2], al[j / 2 + 1], 0x5432);
            const uint32_t p1 = (j & 1) == 0 ? al[j / 2 + 1] : __byte_perm(al[j / 2 + 1], al[j / 2 + 2], 0x5432);
            acc[j] = __dp2a_lo(p0, r, acc[j]);
            acc[j] = __dp2a_hi(p1, r, acc[j]);
        }
    }
}

template <int NS, bool K32, bool BYTE>
__global__ void __launch_bounds__(WARPS * 32, 2) k_match(const MatchParams p, const __grid_constant__ CUtensorMap tmap,
                                                        const __grid_constant__ CUtensorMap emap) {
    using G = Geo<NS>;
    constexpr int R_ = G::R, E = G::E, EC = G::EC, KB = G::KB, UNITS = G::UNITS, ITERS = G::ITERS;

    // tile class: byte tiles belong to the BYTE instantiation, all others to the general one
    const uint32_t cls = p.tcls[p.tile0 + blockIdx.x];
    if (BYTE != (((cls >> 16) & 1u) != 0u)) return;
    const uint32_t tmin = cls & 0xFFFFu;
    const bool narrow = BYTE || ((cls >> 17) & 1u) != 0u;

    extern __shared__ __align__(128) unsigned char s_raw[];
    uint16_t *s_win = reinterpret_cast<uint16_t *>(s_raw);
    uint32_t *s_bw = reinterpret_cast<uint32_t *>(s_raw);  // byte path: packed bytes
    unsigned char *s_tab = s_raw + (BYTE ? G::BWIN_BYTES : G::WIN_BYTES);
    uint32_t *s_s2 = reinterpret_cast<uint32_t *>(s_tab);  // byte kernel: centred energies S2'
    uint2 *s_e = reinterpret_cast<uint2 *>(s_tab);         // general kernel: {S2 mod 2^32, S1 | S2hi << 24}
    __shared__ uint32_t s_surv[WARPS][BYTE ? 2 : 1][CAP];  // byte kernel: one list per reference of a pair
    __shared__ uint32_t s_refhi[BYTE ? 1 : WARPS][16];  // high byte plane of a wide-range reference block

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const B4dGeom &g = p.g;

    long long t = p.tile0 + blockIdx.x;
    const int tx = (int)(t % g.tx);
    t /= g.tx;
    const int ty = (int)(t % g.ty);
    t /= g.ty;
    const int tz = (int)(t % g.tz);
    const int vol = (int)(t / g.tz);
    const int iz0 = tz * 4, iy0 = ty * 4, ix0 = tx * 4;
    const int bz = g.refz[iz0] - R_, by = g.refy[iy0] - R_, bx = g.refx[ix0] - R_;
    const uint16_t *__restrict__ uv = p.u + (long long)vol * g.vol_stride;
    const uint2 *__restrict__ s21v = p.s21 + (long long)vol * g.vol_stride;
    // General kernel: the staged window starts at an EVEN global x when rows are 4-byte aligned
    // (W even), so that it can be filled by 4-byte cp.async; xo = 0 or 1 shifts window columns.
    const int xo = (BYTE || (g.W & 1)) ? 0 : (bx & 1);
    const int xt = bx & 1;  // general kernel: table column of origin bx (the box starts at the even column at or below it)

    if (BYTE) {
        if (p.use_tma) {
            // (1) TMA: the (E x E x E) uint16 neighbourhood as ONE 4-D box load (x extent rounded up to BOXW), issued by
            // one thread, zero fill outside the volume by the tensor map, completion on an mbarrier — no per-element
            // address arithmetic, nothing on the LSU issue path.  It lands dense in the table space.
            __shared__ __align__(8) unsigned long long s_mbar;
            uint16_t *s_tmp = reinterpret_cast<uint16_t *>(s_tab);
            const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&s_mbar);
            if (threadIdx.x == 0) mbar_init(mbar, 1);
            __syncthreads();
            const int xb = bx & 7, bxa = bx - xb;  // box origin: the 16-byte aligned column at or below bx
            if (threadIdx.x == 0) {
                mbar_expect_tx(mbar, G::BOX_BYTES);
                tma_load_4d((uint32_t)__cvta_generic_to_shared(s_tmp), &tmap, mbar, bxa, by, bz, vol);
            }
            mbar_wait(mbar, 0);
            // (2) bytes v - tile_min, four per word (columns past the window hold data no valid candidate reads)
            for (int id = threadIdx.x; id < E * E * G::RW; id += WARPS * 32) {
                const int row = id / G::RW, xw = id - row * G::RW;
                const int z = row / E, y = row - z * E;
                const uint16_t *src = s_tmp + row * G::BOXW + xb + 4 * xw;
                const uint32_t b0 = (src[0] - tmin) & 0xFFu, b1 = (src[1] - tmin) & 0xFFu;
                const uint32_t b2 = (src[2] - tmin) & 0xFFu, b3 = (src[3] - tmin) & 0xFFu;
                s_bw[z * G::PSW + y * G::RSW + xw] = b0 | (b1 << 8) | (b2 << 16) | (b3 << 24);
            }
            __syncthreads();
            // (3) centred block energies from the byte window (as below)
            for (int col = threadIdx.x; col < EC * EC; col += WARPS * 32) {
                const int y = col / EC, x = col - y * EC;
                const uint32_t sel = 0x3210u + 0x1111u * (uint32_t)(x & 3);
                uint32_t r1 = 0u, r2 = 0u, r3 = 0u;
                for (int z = 0; z < E; ++z) {
                    uint32_t r0 = 0u;
#pragma unroll
                    for (int dy = 0; dy < 4; ++dy) {
                        const uint32_t *w = s_bw + z * G::PSW + (y + dy) * G::RSW + (x >> 2);
                        const uint32_t q = __byte_perm(w[0], w[1], sel);
                        r0 = __dp4a(q, q, r0);
                    }
                    if (z >= 3) s_s2[(z - 3) * G::AC + y * G::BC + x] = r0 + r1 + r2 + r3;
                    r3 = r2;
                    r2 = r1;
                    r1 = r0;
                }
            }
        } else if (!(g.W & 1)) {
            // (1) raw uint16 window -> scratch (the S2' table's space) by cp.async, as in the
            // general kernel: even global x origin, zero fill outside the volume
            uint16_t *s_tmp = reinterpret_cast<uint16_t *>(s_tab);
            const uint32_t tmp_base = (uint32_t)__cvta_generic_to_shared(s_tmp);
            const int xb = bx & 1, bxe = bx - xb;
            for (int id = threadIdx.x; id < E * E * G::BW; id += WARPS * 32) {
                const int row = id / G::BW, c = id - row * G::BW;
                const int z = row / E, y = row - z * E;
                const int gz = bz + z, gy = by + y, gxc = bxe + 2 * c;
                const bool in = (unsigned)gz < (unsigned)g.D && (unsigned)gy < (unsigned)g.H &&
                                (unsigned)gxc < (unsigned)g.W;
                const uint16_t *src = in ? uv + ((long long)gz * g.H + gy) * g.W + gxc : uv;
                cp_async4_zfill(tmp_base + 4u * (uint32_t)(z * G::AW + y * G::BW + c), src, in ? 4u : 0u);
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncthreads();
            // (2) bytes v - tile_min, four per word (voxels outside the volume give junk bytes that
            // no valid candidate reads)
            for (int id = threadIdx.x; id < E * E * G::RW; id += WARPS * 32) {
                const int row = id / G::RW, xw = id - row * G::RW;
                const int z = row / E, y = row - z * E;
                const uint16_t *src = s_tmp + z * G::SZ + y * G::SY + xb + 4 * xw;
                const uint32_t b0 = (src[0] - tmin) & 0xFFu, b1 = (src[1] - tmin) & 0xFFu;
                const uint32_t b2 = (src[2] - tmin) & 0xFFu, b3 = (src[3] - tmin) & 0xFFu;
                s_bw[z * G::PSW + y * G::RSW + xw] = b0 | (b1 << 8) | (b2 << 16) | (b3 << 24);
            }
            __syncthreads();
            // (3) centred block energies S2'(z,y,x) = sum over the 4x4x4 block of byte^2, from the
            // byte window: one thread per (y, x) column marches along z with a 4-plane sliding sum
            for (int col = threadIdx.x; col < EC * EC; col += WARPS * 32) {
                const int y = col / EC, x = col - y * EC;
                const uint32_t sel = 0x3210u + 0x1111u * (uint32_t)(x & 3);
                uint32_t r1 = 0u, r2 = 0u, r3 = 0u;  // plane sums of z-1, z-2, z-3
                for (int z = 0; z < E; ++z) {
                    uint32_t r0 = 0u;
#pragma unroll
                    for (int dy = 0; dy < 4; ++dy) {
                        const uint32_t *w = s_bw + z * G::PSW + (y + dy) * G::RSW + (x >> 2);
                        const uint32_t q = __byte_perm(w[0], w[1], sel);
                        r0 = __dp4a(q, q, r0);
                    }
                    if (z >= 3) s_s2[(z - 3) * G::AC + y * G::BC + x] = r0 + r1 + r2 + r3;
                    r3 = r2;
                    r2 = r1;
                    r1 = r0;
                }
            }
        } else {
        // odd row length: rows are not 4-byte aligned -> plain loads, one row per warp iteration
        const int gx = bx + lane;
        const bool xin = lane < E && (unsigned)gx < (unsigned)g.W;
#pragma unroll 4
        for (int row = warp; row < E * E; row += WARPS) {
            const int z = row / E, y = row - z * E;
            const int gz = bz + z, gy = by + y;
            uint32_t v = 0;
            const bool in = xin && (unsigned)gz < (unsigned)g.D && (unsigned)gy < (unsigned)g.H;
            if (in) v = uv[((long long)gz * g.H + gy) * g.W + gx];
            // bytes v - tile_min (0 outside the volume), four per word
            uint32_t bt = in ? ((v - tmin) & 0xFFu) : 0u;
            bt |= __shfl_down_sync(B4D_FULL, bt, 1) << 8;
            bt |= __shfl_down_sync(B4D_FULL, bt, 2) << 16;
            if ((lane & 3) == 0 && lane < 4 * G::RW) s_bw[z * G::PSW + y * G::RSW + (lane >> 2)] = bt;
        }
        const bool cin = lane < EC && (unsigned)gx <= (unsigned)(g.W - 4);
        const uint32_t m2 = 2u * tmin, m64 = 64u * tmin * tmin;
#pragma unroll 4
        for (int row = warp; row < EC * EC; row += WARPS) {
            const int z = row / EC, y = row - z * EC;
            const int gz = bz + z, gy = by + y;
            uint2 v = make_uint2(0u, 0u);
            if (cin && (unsigned)gz <= (unsigned)(g.D - 4) && (unsigned)gy <= (unsigned)(g.H - 4))
                v = s21v[((long long)gz * g.H + gy) * g.W + gx];
            // centred block energies S2' = S2 - 2 m S1 + 64 m^2 (exact: S2' <= 64 * 255^2)
            if (lane < EC)
                s_s2[z * G::AC + y * G::BC + lane] = (v.x | v.y) ? v.x - m2 * (v.y & 0xFFFFFFu) + m64 : 0u;
        }
        }
    } else {
        // Asynchronous staging (cp.async, zero fill outside the volume): no register round trip,
        // every copy of the tile in flight at once, one wait.
        const uint32_t win_base = (uint32_t)__cvta_generic_to_shared(s_win);
        const uint32_t tab_base = (uint32_t)__cvta_generic_to_shared(s_e);
        if (!(g.W & 1)) {
            const int bxe = bx - xo;  // even
            for (int id = threadIdx.x; id < E * E * G::BW; id += WARPS * 32) {
                const int row = id / G::BW, c = id - row * G::BW;
                const int z = row / E, y = row - z * E;
                const int gz = bz + z, gy = by + y, gxc = bxe + 2 * c;
                const bool in = (unsigned)gz < (unsigned)g.D && (unsigned)gy < (unsigned)g.H &&
                                (unsigned)gxc < (unsigned)g.W;  // gxc and W even: the pair is inside
                const uint16_t *src = in ? uv + ((long long)gz * g.H + gy) * g.W + gxc : uv;
                cp_async4_zfill(win_base + 4u * (uint32_t)(z * G::AW + y * G::BW + c), src, in ? 4u : 0u);
            }
        } else {  // odd row length: rows are not 4-byte aligned, plain loads
            for (int id = threadIdx.x; id < E * E * E; id += WARPS * 32) {
                const int x = id % E, y = (id / E) % E, z = id / (E * E);
                const int gz = bz + z, gy = by + y, gx = bx + x;
                uint32_t v = 0;
                if ((unsigned)gz < (unsigned)g.D && (unsigned)gy < (unsigned)g.H && (unsigned)gx < (unsigned)g.W)
                    v = uv[((long long)gz * g.H + gy) * g.W + gx];
                s_win[z * G::SZ + y * G::SY + x] = (uint16_t)v;
            }
        }
        if (p.use_tma_tab) {
            // the whole table as ONE box load (the map only spans valid block origins, everything else arrives as zero)
            __shared__ __align__(8) unsigned long long s_mbar_e;
            const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&s_mbar_e);
            if (threadIdx.x == 0) {
                mbar_init(mbar, 1);
                mbar_expect_tx(mbar, G::TAB_BOX_BYTES);
                tma_load_4d(tab_base, &emap, mbar, bx - xt, by, bz, vol);
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncthreads();  // the barrier is initialised for everybody
            mbar_wait(mbar, 0);
        } else {
            for (int id = threadIdx.x; id < EC * EC * EC; id += WARPS * 32) {
                const int x = id % EC, y = (id / EC) % EC, z = id / (EC * EC);
                const int gz = bz + z, gy = by + y, gx = bx + x;
                const bool in = (unsigned)gz <= (unsigned)(g.D - 4) && (unsigned)gy <= (unsigned)(g.H - 4) &&
                                (unsigned)gx <= (unsigned)(g.W - 4);
                const uint2 *src = in ? s21v + ((long long)gz * g.H + gy) * g.W + gx : s21v;
                cp_async8_zfill(tab_base + 8u * (uint32_t)(z * G::TAC + y * G::TBW + x + xt), src, in ? 8u : 0u);
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
        }
    }
    __syncthreads();
    if (!narrow && threadIdx.x == 0 && p.stats) atomicAdd(&p.stats[1], 1ull);
    if (BYTE && threadIdx.x == 0 && p.stats) atomicAdd(&p.stats[3], 1ull);

    const int K = p.K;
    const uint32_t tau = p.tau;
    // A candidate is acceptable iff its key is <= KEYMAX (SSD <= tau): where no other test is needed the keys are
    // built without the tau comparison — the SSD is saturated to the key's field instead (one min instead of a
    // compare and a select) — and every bound starts at KEYMAX.
    const uint32_t DMAX = (1u << (32 - KB)) - 1u;
    const uint32_t KEYMAX = (min(tau, DMAX - 1u) << KB) | ((1u << KB) - 1u);

    // ---- byte tiles whose four reference columns are regular: two references per pass (neighbours in x).  Only the
    // common case runs here (one pass, bound refined on the fly); a pair whose survivor list overflows is left to
    // the one-reference loop below (redo mask).
    uint32_t redo = 0u;
    const bool pair_tile = BYTE && ((cls >> 18) & 1u) != 0u;
    if constexpr (BYTE) {
        if (pair_tile) {
#pragma unroll 1
            for (int pr = warp; pr < 32; pr += WARPS) {
                const int iz = iz0 + (pr >> 3), iy = iy0 + ((pr >> 1) & 3), ixa = ix0 + 2 * (pr & 1);
                if (iz >= g.nrz || iy >= g.nry) continue;  // warp-uniform
                const int oz = g.refz[iz], oy = g.refy[iy], oxa = g.refx[ixa];
                const int wz0 = oz - R_ - bz, wy0 = oy - R_ - by, wx0 = oxa - R_ - bx;
                uint32_t refa[16], refb[16];
                {
                    const int rxa = wx0 + R_, rxb = rxa + 3;
                    const uint32_t sa = 0x3210u + 0x1111u * (uint32_t)(rxa & 3), sb = 0x3210u + 0x1111u * (uint32_t)(rxb & 3);
#pragma unroll
                    for (int z = 0; z < 4; ++z)
#pragma unroll
                        for (int y = 0; y < 4; ++y) {
                            const uint32_t *row = s_bw + (wz0 + R_ + z) * G::PSW + (wy0 + R_ + y) * G::RSW;
                            refa[z * 4 + y] = __byte_perm(row[rxa >> 2], row[(rxa >> 2) + 1], sa);
                            refb[z * 4 + y] = __byte_perm(row[rxb >> 2], row[(rxb >> 2) + 1], sb);
                        }
                }
                const uint32_t *e_ref = s_s2 + (wz0 + R_) * G::AC + (wy0 + R_) * G::BC + (wx0 + R_);
                const uint32_t s2a = e_ref[0], s2b = e_ref[3];
                const uint32_t bsel = 0x3210u + 0x1111u * (uint32_t)(wx0 & 3);
                const int jloa = max(0, R_ - oxa), jhia = min(NS - 1, g.W - 4 - oxa + R_);
                const int jlob = max(0, R_ - oxa - 3), jhib = min(NS - 1, g.W - 4 - oxa - 3 + R_);
                const bool xfull = jloa == 0 && jlob == 0 && jhia == NS - 1 && jhib == NS - 1;
                const long long rlina = (long long)vol * g.refs_per_vol + ((long long)iz * g.nry + iy) * g.nrx + ixa;
                uint32_t la1 = B4D_INVALID_KEY, la2 = B4D_INVALID_KEY, lb1 = B4D_INVALID_KEY, lb2 = B4D_INVALID_KEY;
                uint32_t Ba = KEYMAX, Bb = KEYMAX;
                int na = 0, nb = 0;  // survivor counts (warp-uniform)
                __syncwarp();
#pragma unroll 1
                for (int it = 0; it < ITERS; ++it) {
                    const int unit = (int)((G::ORDER >> (4 * it)) & 15ull) * 32 + lane;
                    const int dz = unit / NS, dy = unit - dz * NS;
                    const int cz = oz - R_ + dz, cy = oy - R_ + dy;
                    const bool uvalid = unit < UNITS && cz >= 0 && cz <= g.D - 4 && cy >= 0 && cy <= g.H - 4;
                    if (!__any_sync(B4D_FULL, uvalid)) continue;
                    uint32_t ka[NS], kb[NS];
#pragma unroll
                    for (int j = 0; j < NS; ++j) ka[j] = kb[j] = B4D_INVALID_KEY;
                    if (uvalid) {
                        uint32_t acca[NS], accb[NS];
                        bcorr_row_pair<NS>(s_bw + (wz0 + dz) * G::PSW + (wy0 + dy) * G::RSW + (wx0 >> 2), bsel, refa, refb, acca,
                                           accb);
                        const uint32_t *e = s_s2 + (wz0 + dz) * G::AC + (wy0 + dy) * G::BC + wx0;
                        if (xfull) {  // warp-uniform: every dx of both windows is inside the volume (all but the edge tiles)
#pragma unroll
                            for (int j = 0; j < NS; ++j) {
                                const uint32_t idx = (uint32_t)(unit * NS + j);
                                const uint32_t da = min((e[j] + s2a) - 2u * acca[j], DMAX);
                                ka[j] = mad_key(da, 1u << KB, idx);
                                const uint32_t db = min((e[j + 3] + s2b) - 2u * accb[j], DMAX);
                                kb[j] = mad_key(db, 1u << KB, idx);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < NS; ++j) {
                                const uint32_t idx = (uint32_t)(unit * NS + j);
                                const uint32_t da = (e[j] + s2a) - 2u * acca[j];
                                const bool oka = da <= tau && j >= jloa && j <= jhia;
                                ka[j] = oka ? mad_key(da, 1u << KB, idx) : B4D_INVALID_KEY;
                                const uint32_t db = (e[j + 3] + s2b) - 2u * accb[j];
                                const bool okb = db <= tau && j >= jlob && j <= jhib;
                                kb[j] = okb ? mad_key(db, 1u << KB, idx) : B4D_INVALID_KEY;
                            }
                        }
                    }
#pragma unroll
                    for (int j = 0; j < NS; ++j) {
                        if (K32) {
                            la2 = min(la2, max(la1, ka[j]));
                            lb2 = min(lb2, max(lb1, kb[j]));
                        }
                        la1 = min(la1, ka[j]);
                        lb1 = min(lb1, kb[j]);
                    }
                    Ba = min(Ba, kth_smallest32(K32 ? la2 : la1, K32 ? 15 : K - 1, lane));
                    Bb = min(Bb, kth_smallest32(K32 ? lb2 : lb1, K32 ? 15 : K - 1, lane));
                    const unsigned below = (1u << lane) - 1u;
#pragma unroll
                    for (int j = 0; j < NS; ++j) {
                        const bool ta = ka[j] <= Ba, tb = kb[j] <= Bb;
                        const unsigned ma = __ballot_sync(B4D_FULL, ta), mb = __ballot_sync(B4D_FULL, tb);
                        const int pa = na + __popc(ma & below), pb = nb + __popc(mb & below);
                        if (ta && pa < CAP) s_surv[warp][0][pa] = ka[j];
                        if (tb && pb < CAP) s_surv[warp][1][pb] = kb[j];
                        na += __popc(ma);
                        nb += __popc(mb);
                    }
                }
                __syncwarp();
                if (na > CAP || nb > CAP) {  // rare: both references go through the one-reference loop
                    redo |= 1u << pr;
                    continue;
                }
#pragma unroll 1
                for (int sref = 0; sref < 2; ++sref) {
                    uint32_t *lst = s_surv[warp][sref];
                    const int n = sref ? nb : na;
                    const uint32_t B = sref ? Bb : Ba;
                    const long long rlin = rlina + sref;
                    // compact the survivors that are <= the final bound, then rank-sort them (as below)
                    uint32_t mine[CAP / 32];
#pragma unroll
                    for (int s = 0; s < CAP / 32; ++s) {
                        const int e = s * 32 + lane;
                        uint32_t k = (e < n) ? lst[e] : B4D_INVALID_KEY;
                        mine[s] = (k > B) ? B4D_INVALID_KEY : k;
                    }
                    __syncwarp();
                    int nf = 0;
#pragma unroll
                    for (int s = 0; s < CAP / 32; ++s) {
                        if (s * 32 >= n) break;  // warp-uniform
                        const bool keep = mine[s] != B4D_INVALID_KEY;
                        const unsigned bal = __ballot_sync(B4D_FULL, keep);
                        if (keep) lst[nf + __popc(bal & ((1u << lane) - 1u))] = mine[s];
                        nf += __popc(bal);
                    }
                    __syncwarp();
                    const int ns = min(nf, K);
                    const int kp = ns > 0 ? (1 << (31 - __clz(ns))) : 0;
                    for (int s0 = 0; s0 < nf; s0 += 64) {
                        const int e0 = s0 + lane, e1 = s0 + 32 + lane;
                        const uint32_t k0 = e0 < nf ? lst[e0] : B4D_INVALID_KEY;
                        const uint32_t k1 = e1 < nf ? lst[e1] : B4D_INVALID_KEY;
                        int r0 = 0, r1 = 0;
                        for (int e = 0; e < nf; ++e) {
                            const uint32_t o = lst[e];
                            r0 += (o < k0) ? 1 : 0;
                            r1 += (o < k1) ? 1 : 0;
                        }
                        if (k0 != B4D_INVALID_KEY && r0 < kp) {
                            p.widx[rlin * K + r0] = (uint16_t)(k0 & ((1u << KB) - 1u));
                            if (p.ssd_out) p.ssd_out[rlin * K + r0] = k0 >> KB;
                        }
                        if (k1 != B4D_INVALID_KEY && r1 < kp) {
                            p.widx[rlin * K + r1] = (uint16_t)(k1 & ((1u << KB) - 1u));
                            if (p.ssd_out) p.ssd_out[rlin * K + r1] = k1 >> KB;
                        }
                    }
                    if (lane == 0) p.cnt[rlin] = (uint8_t)kp;
                    __syncwarp();
                }
            }
            if (redo == 0u) return;  // warp-uniform: nothing left for this warp
        }
    }

    for (int q8 = 0; q8 < 64 / WARPS; ++q8) {
        // reference index of this warp's q8-th turn: plain tiles, rr = warp + 8 q8; pair tiles, the two references
        // of the warp's pairs that asked for a second go
        const int rr = pair_tile ? 2 * (warp + WARPS * (q8 >> 1)) + (q8 & 1) : warp + WARPS * q8;
        if (pair_tile && ((redo >> (rr >> 1)) & 1u) == 0u) continue;
        const int iz = iz0 + (rr >> 4), iy = iy0 + ((rr >> 2) & 3), ix = ix0 + (rr & 3);
        if (iz >= g.nrz || iy >= g.nry || ix >= g.nrx) continue;  // warp-uniform
        const int oz = g.refz[iz], oy = g.refy[iy], ox = g.refx[ix];
        const int wz0 = oz - R_ - bz, wy0 = oy - R_ - by, wx0 = ox - R_ - bx;  // window origin in the tile
        const int wxw = wx0 + xo;  // window column of the search-window origin
        const uint16_t *refp = s_win + (wz0 + R_) * G::SZ + (wy0 + R_) * G::SY + (wxw + R_);
        // reference block as bytes, one word per block row: BYTE kernel v - tile_min; general kernel
        // the low bytes of r - r_min (the high bytes, when the block spans more than 255 counts,
        // go to shared memory)
        uint32_t refw[16];
        uint32_t s2ref = 0;
        uint32_t rmin = 0, s1ref = 0;
        int npass = 1;
        const uint32_t bsel = 0x3210u + 0x1111u * (uint32_t)(wx0 & 3);  // PRMT selector of the row alignment
        if constexpr (BYTE) {
            const int rx = wx0 + R_;
            const uint32_t rsel = 0x3210u + 0x1111u * (uint32_t)(rx & 3);
#pragma unroll
            for (int z = 0; z < 4; ++z)
#pragma unroll
                for (int y = 0; y < 4; ++y) {
                    const uint32_t *rw = s_bw + (wz0 + R_ + z) * G::PSW + (wy0 + R_ + y) * G::RSW + (rx >> 2);
                    refw[z * 4 + y] = __byte_perm(rw[0], rw[1], rsel);
                }
            s2ref = s_s2[(wz0 + R_) * G::AC + (wy0 + R_) * G::BC + (wx0 + R_)];
        } else {
            {
                // range of the reference block: lanes read two voxels each
                const uint32_t va = refp[(lane >> 4) * G::SZ + ((lane >> 2) & 3) * G::SY + (lane & 3)];
                const uint32_t vb = refp[(2 + (lane >> 4)) * G::SZ + ((lane >> 2) & 3) * G::SY + (lane & 3)];
                rmin = __reduce_min_sync(B4D_FULL, min(va, vb));
                const uint32_t rmax = __reduce_max_sync(B4D_FULL, max(va, vb));
                npass = (rmax - rmin <= 255u) ? 1 : 2;  // r - r_min < 2^16: low and high byte planes
                const uint2 er = s_e[(wz0 + R_) * G::TAC + (wy0 + R_) * G::TBW + (wx0 + R_) + xt];
                s2ref = er.x;
                s1ref = er.y;
                // byte planes of r - r_min, one word per block row: every lane already holds two voxels (rows
                // lane >> 2 and 8 + (lane >> 2)); the four bytes of a row are packed by two shuffles, lane 4 r then holds
                // the word of row r and hands it to everybody
                const uint32_t da = va - rmin, db = vb - rmin;
                uint32_t la = da & 0xFFu, lb = db & 0xFFu;
                la |= __shfl_down_sync(B4D_FULL, la, 1) << 8;
                lb |= __shfl_down_sync(B4D_FULL, lb, 1) << 8;
                la |= __shfl_down_sync(B4D_FULL, la, 2) << 16;
                lb |= __shfl_down_sync(B4D_FULL, lb, 2) << 16;
#pragma unroll
                for (int r8 = 0; r8 < 8; ++r8) {
                    refw[r8] = __shfl_sync(B4D_FULL, la, 4 * r8);
                    refw[8 + r8] = __shfl_sync(B4D_FULL, lb, 4 * r8);
                }
                if (npass == 2) {  // warp-uniform
                    uint32_t ha = da >> 8, hb = db >> 8;
                    ha |= __shfl_down_sync(B4D_FULL, ha, 1) << 8;
                    hb |= __shfl_down_sync(B4D_FULL, hb, 1) << 8;
                    ha |= __shfl_down_sync(B4D_FULL, ha, 2) << 16;
                    hb |= __shfl_down_sync(B4D_FULL, hb, 2) << 16;
                    if ((lane & 3) == 0) {
                        s_refhi[warp][lane >> 2] = ha;
                        s_refhi[warp][8 + (lane >> 2)] = hb;
                    }
                }
                __syncwarp();
            }
        }
        // valid dx range of candidates: cx = ox - R_ + j in [0, W-4]
        const int jlo = max(0, R_ - ox), jhi = min(NS - 1, g.W - 4 - ox + R_);
        const bool xfull = jlo == 0 && jhi == NS - 1;

        const long long rlin = (long long)vol * g.refs_per_vol + ((long long)iz * g.nry + iy) * g.nrx + ix;

        // mode 0: one pass, bound refined on the fly.  mode 1 (survivor list overflowed):
        // one more pass with the final bound of mode 0 fixed from the start.  mode 2 (still
        // overflowing): K rounds of "smallest key greater than the previous one".
        int mode = 0;
        uint32_t Bfix = KEYMAX;
        uint32_t prev = 0;                 // mode 2: last extracted key
        int nsel = 0;                      // mode 2: keys extracted so far
        uint32_t mykey = B4D_INVALID_KEY;  // mode 2: lane k holds the k-th key
        for (;;) {
            uint32_t lmin1 = B4D_INVALID_KEY, lmin2 = B4D_INVALID_KEY;
            uint32_t B = Bfix;
            int nsurv = 0;  // survivor count of this warp (uniform; the list is warp-private)
            __syncwarp();
#pragma unroll 1
            for (int it = 0; it < ITERS; ++it) {
                const int unit = (int)((G::ORDER >> (4 * it)) & 15ull) * 32 + lane;
                const int dz = unit / NS, dy = unit - dz * NS;
                const int cz = oz - R_ + dz, cy = oy - R_ + dy;
                const bool uvalid = unit < UNITS && cz >= 0 && cz <= g.D - 4 && cy >= 0 && cy <= g.H - 4;
                if (!__any_sync(B4D_FULL, uvalid)) continue;
                uint32_t key[NS];
#pragma unroll
                for (int j = 0; j < NS; ++j) key[j] = B4D_INVALID_KEY;
                if constexpr (BYTE) {
                    if (uvalid) {
                        uint32_t acc[NS];
                        bcorr_row<NS>(s_bw + (wz0 + dz) * G::PSW + (wy0 + dy) * G::RSW + (wx0 >> 2), bsel, refw, acc);
                        const uint32_t *e = s_s2 + (wz0 + dz) * G::AC + (wy0 + dy) * G::BC + wx0;
#pragma unroll
                        for (int j = 0; j < NS; ++j) {
                            const uint32_t ssd = (e[j] + s2ref) - 2u * acc[j];
                            const bool ok = ssd <= tau && (xfull || (j >= jlo && j <= jhi));
                            key[j] = ok ? mad_key(ssd, 1u << KB, (uint32_t)(unit * NS + j)) : B4D_INVALID_KEY;
                        }
                    }
                } else {
                    if (uvalid) {
                        // sum(a r) = sum(a rl) + 256 sum(a rh) + r_min S1(a): one IDP.2A pass per
                        // reference byte plane (each pass < 2^31)
                        const int pp = wxw & 1;
                        const uint32_t *wb = reinterpret_cast<const uint32_t *>(s_win) +
                                             (((wz0 + dz) * G::SZ + (wy0 + dy) * G::SY + wxw - pp) >> 1);
                        const uint32_t psel = pp ? 0x5432u : 0x3210u;
                        uint32_t acc[NS], acch[NS];
                        r8corr_row<NS>(wb, psel, refw, acc);
                        if (npass == 2) {
                            r8corr_row_rolled<NS>(wb, psel, s_refhi[warp], acch);
                        } else {
#pragma unroll
                            for (int j = 0; j < NS; ++j) acch[j] = 0u;
                        }
                        const uint2 *e = s_e + (wz0 + dz) * G::TAC + (wy0 + dy) * G::TBW + wx0 + xt;
                        if (narrow) {
                            // everything modulo 2^32: exact because the true SSD < 2^32 on a narrow tile
                            const uint32_t rm2 = 2u * rmin;
                            if (xfull) {  // warp-uniform: no candidate of this window leaves the volume along x
#pragma unroll
                                for (int j = 0; j < NS; ++j) {
                                    const uint2 ev = e[j];
                                    const uint32_t dot = acc[j] + (acch[j] << 8);
                                    const uint32_t ssd = min((ev.x + s2ref) - 2u * dot - rm2 * (ev.y & 0xFFFFFFu), DMAX);
                                    key[j] = mad_key(ssd, 1u << KB, (uint32_t)(unit * NS + j));
                                }
                            } else {
#pragma unroll
                                for (int j = 0; j < NS; ++j) {
                                    const uint2 ev = e[j];
                                    const uint32_t dot = acc[j] + (acch[j] << 8);
                                    const uint32_t ssd = (ev.x + s2ref) - 2u * dot - rm2 * (ev.y & 0xFFFFFFu);
                                    const bool ok = ssd <= tau && j >= jlo && j <= jhi;
                                    key[j] = ok ? mad_key(ssd, 1u << KB, (uint32_t)(unit * NS + j)) : B4D_INVALID_KEY;
                                }
                            }
                        } else {
                            // wide tile: the same sums, combined exactly in 64 bits
                            const unsigned long long s2r = (unsigned long long)s2ref | ((unsigned long long)(s1ref >> 24) << 32);
#pragma unroll
                            for (int j = 0; j < NS; ++j) {
                                const uint2 ev = e[j];
                                const uint32_t e1j = ev.y;
                                const unsigned long long s2a = (unsigned long long)ev.x | ((unsigned long long)(e1j >> 24) << 32);
                                const unsigned long long dot = (unsigned long long)acc[j] + ((unsigned long long)acch[j] << 8) +
                                                               (unsigned long long)rmin * (e1j & 0xFFFFFFu);
                                const unsigned long long ssd = s2a + s2r - 2ull * dot;
                                const bool ok = ssd <= (unsigned long long)tau && j >= jlo && j <= jhi;
                                key[j] = ok ? mad_key((uint32_t)ssd, 1u << KB, (uint32_t)(unit * NS + j)) : B4D_INVALID_KEY;
                            }
                        }
                    }
                }
                if (mode < 2) {
                    if (mode == 0) {
#pragma unroll
                        for (int j = 0; j < NS; ++j) {
                            if (K32) lmin2 = min(lmin2, max(lmin1, key[j]));
                            lmin1 = min(lmin1, key[j]);
                        }
                        const uint32_t b = kth_smallest32(K32 ? lmin2 : lmin1, K32 ? 15 : K - 1, lane);
                        B = min(B, b);
                    }
#pragma unroll
                    for (int j = 0; j < NS; ++j) {
                        const bool take = key[j] <= B;
                        const unsigned m = __ballot_sync(B4D_FULL, take);
                        const int pos = nsurv + __popc(m & ((1u << lane) - 1u));
                        if (take && pos < CAP) s_surv[warp][0][pos] = key[j];
                        nsurv += __popc(m);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < NS; ++j) {
                        const uint32_t k = ((nsel == 0 || key[j] > prev) && key[j] <= KEYMAX) ? key[j] : B4D_INVALID_KEY;
                        lmin1 = min(lmin1, k);
                    }
                }
            }
            __syncwarp();
            if (mode < 2) {
                const int n = nsurv;
                if (n <= CAP) {
                    // compact the survivors that are <= the final bound, then rank-sort them
                    uint32_t mine[CAP / 32];
#pragma unroll
                    for (int s = 0; s < CAP / 32; ++s) {
                        const int e = s * 32 + lane;
                        uint32_t k = (e < n) ? s_surv[warp][0][e] : B4D_INVALID_KEY;
                        mine[s] = (k > B) ? B4D_INVALID_KEY : k;
                    }
                    __syncwarp();
                    int nf = 0;
#pragma unroll
                    for (int s = 0; s < CAP / 32; ++s) {
                        if (s * 32 >= n) break;  // warp-uniform
                        const bool keep = mine[s] != B4D_INVALID_KEY;
                        const unsigned bal = __ballot_sync(B4D_FULL, keep);
                        if (keep) s_surv[warp][0][nf + __popc(bal & ((1u << lane) - 1u))] = mine[s];
                        nf += __popc(bal);
                    }
                    __syncwarp();
                    const int ns = min(nf, K);
                    const int kp = ns > 0 ? (1 << (31 - __clz(ns))) : 0;
                    for (int s0 = 0; s0 < nf; s0 += 64) {
                        const int e0 = s0 + lane, e1 = s0 + 32 + lane;
                        const uint32_t k0 = e0 < nf ? s_surv[warp][0][e0] : B4D_INVALID_KEY;
                        const uint32_t k1 = e1 < nf ? s_surv[warp][0][e1] : B4D_INVALID_KEY;
                        int r0 = 0, r1 = 0;
                        for (int e = 0; e < nf; ++e) {
                            const uint32_t o = s_surv[warp][0][e];
                            r0 += (o < k0) ? 1 : 0;
                            r1 += (o < k1) ? 1 : 0;
                        }
                        if (k0 != B4D_INVALID_KEY && r0 < kp) {
                            p.widx[rlin * K + r0] = (uint16_t)(k0 & ((1u << KB) - 1u));
                            if (p.ssd_out) p.ssd_out[rlin * K + r0] = k0 >> KB;
                        }
                        if (k1 != B4D_INVALID_KEY && r1 < kp) {
                            p.widx[rlin * K + r1] = (uint16_t)(k1 & ((1u << KB) - 1u));
                            if (p.ssd_out) p.ssd_out[rlin * K + r1] = k1 >> KB;
                        }
                    }
                    if (lane == 0) p.cnt[rlin] = (uint8_t)kp;
                    break;
                }
                // list overflowed: retry once with the (tightest) final bound, then go exact-but-slow
                if (lane == 0 && p.stats) atomicAdd(&p.stats[mode == 0 ? 0 : 2], 1ull);
                Bfix = B;
                ++mode;
                continue;
            }
            // mode 2 round finished: lmin1 = smallest key > prev in this lane
            const uint32_t m = warp_min_u32(lmin1);
            if (m != B4D_INVALID_KEY) {
                if (lane == nsel) mykey = m;
                prev = m;
                ++nsel;
            }
            if (m == B4D_INVALID_KEY || nsel == K) {
                const int kp = nsel > 0 ? (1 << (31 - __clz(nsel))) : 0;
                if (lane < kp) {
                    p.widx[rlin * K + lane] = (uint16_t)(mykey & ((1u << KB) - 1u));
                    if (p.ssd_out) p.ssd_out[rlin * K + lane] = mykey >> KB;
                }
                if (lane == 0) p.cnt[rlin] = (uint8_t)kp;
                break;
            }
        }
        __syncwarp();
    }
}

// Tensor map of the uint16 matching image as a 4-D tensor (x, y, z, volume); box = the staged neighbourhood of one
// tile.  Needs row and plane pitches that are multiples of 16 bytes (W % 8 == 0); otherwise the kernels keep the
// cp.async / plain-load staging.  The encoder comes from the driver through the runtime (no -lcuda).
template <int NS>
bool make_window_map(const MatchParams &p, CUtensorMap *map) {
    using G = Geo<NS>;
    std::memset(map, 0, sizeof(*map));
    const B4dGeom &g = p.g;
    if ((g.W & 7) != 0 || getenv("B4D_NO_TMA")) return false;
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)g.W, (cuuint64_t)g.H, (cuuint64_t)g.D, (cuuint64_t)g.nvol};
    const cuuint64_t strides[3] = {(cuuint64_t)g.W * 2, (cuuint64_t)g.W * g.H * 2, (cuuint64_t)g.vol_stride * 2};
    const cuuint32_t box[4] = {(cuuint32_t)G::BOXW, (cuuint32_t)G::E, (cuuint32_t)G::E, 1u};
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<uint16_t *>(p.u), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int NS, bool K32>
void launch_k(const MatchParams &pin, long long tile0, long long tile1, cudaStream_t s) {
    using G = Geo<NS>;
    MatchParams p = pin;
    p.tile0 = tile0;
    CUtensorMap tmap;
    p.use_tma = make_window_map<NS>(p, &tmap) ? 1 : 0;
    CUtensorMap emap;
    std::memset(&emap, 0, sizeof(emap));
    p.use_tma_tab = 0;
    if ((p.g.W & 1) == 0 && !getenv("B4D_NO_TMA") && p.g.D >= 4 && p.g.H >= 4 && p.g.W >= 4) {
        EncodeTiledFn fn = encode_fn();
        // only valid block origins are inside the tensor: extents (W - 3, H - 3, D - 3), true pitches
        const cuuint64_t dims[4] = {(cuuint64_t)(p.g.W - 3), (cuuint64_t)(p.g.H - 3), (cuuint64_t)(p.g.D - 3), (cuuint64_t)p.g.nvol};
        const cuuint64_t strides[3] = {(cuuint64_t)p.g.W * 8, (cuuint64_t)p.g.W * p.g.H * 8, (cuuint64_t)p.g.vol_stride * 8};
        const cuuint32_t box[4] = {(cuuint32_t)G::TBW, (cuuint32_t)G::EC, (cuuint32_t)G::EC, 1u};
        const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
        if (fn && fn(&emap, CU_TENSOR_MAP_DATA_TYPE_UINT64, 4, const_cast<uint2 *>(p.s21), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
            p.use_tma_tab = 1;
    }
    const unsigned tiles = (unsigned)(tile1 - tile0);
    // byte tiles first (cheap), then everything else; each kernel exits at once on a foreign tile
    cudaFuncSetAttribute(k_match<NS, K32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM_B);
    b4d_launch(k_match<NS, K32, true>, tiles, WARPS * 32, G::SMEM_B, s, p, tmap, emap);
    cudaFuncSetAttribute(k_match<NS, K32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM);
    b4d_launch(k_match<NS, K32, false>, tiles, WARPS * 32, G::SMEM, s, p, tmap, emap);
}
// cell planes [cz0, cz1) (min/max table) and tiles [tile0, tile1) (classification + both matcher
// kernels); the whole volume in one go is cz = [0, cd), tiles = [0, all)
template <int NS>
void launch_ns(const MatchParams &p, int cz0, int cz1, long long tile0, long long tile1, cudaStream_t s) {
    // cz0, cz1 count 4-plane layers (the callers' unit): voxel planes [4 cz0, min(4 cz1, D))
    const int z0 = 4 * cz0, z1 = std::min(4 * cz1, p.g.D);
    if (z1 > z0)
        b4d_launch(k_plane_ranges<NS>, (unsigned)((long long)p.g.nvol * (z1 - z0) * p.g.ty), 256, 0, s, p.u, p.g,
                   p.cells, z0, z1);
    if (tile1 > tile0) {
        b4d_launch(k_tile_class<NS>, (unsigned)((tile1 - tile0 + 7) / 8), 256, 0, s, p.cells, p.g, p.tcls, tile0,
                   tile1);
        if (p.K > 16) launch_k<NS, true>(p, tile0, tile1, s);
        else launch_k<NS, false>(p, tile0, tile1, s);
    }
}

}  // namespace

void b4d_launch_block_energy_range(const uint16_t *u, uint2 *s21, int D, int H, int W, int nvol, int zo0, int zo1,
                                   cudaStream_t s) {
    if (zo1 <= zo0) return;
    const long long nzc = (zo1 - zo0 + K0_ZC - 1) / K0_ZC;
    EncodeTiledFn fn = ((W & 7) == 0 && !getenv("B4D_NO_TMA")) ? encode_fn() : nullptr;
    if (fn) {
        CUtensorMap map;
        const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)nvol};
        const cuuint64_t strides[3] = {(cuuint64_t)W * 2, (cuuint64_t)W * H * 2, (cuuint64_t)W * H * D * 2};
        const cuuint32_t box[4] = {(cuuint32_t)K0T_BOXW, (cuuint32_t)K0T_ROWS, 1u, 1u};
        const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
        if (fn(&map, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<uint16_t *>(u), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS) {
            const long long blocks = (long long)((W - 3 + K0T_TX - 1) / K0T_TX) * ((H - 3 + K0_TY - 1) / K0_TY) * nzc * nvol;
            b4d_launch(k_block_energy_tma, (unsigned)blocks, K0T_WARPS * 32, 0, s, map, s21, D, H, W, nvol, zo0, zo1);
            return;
        }
    }
    const long long warps = (long long)((W - 3 + K0_TX - 1) / K0_TX) * ((H - 3 + K0_TY - 1) / K0_TY) * nzc * nvol;
    const long long blocks = (warps + K0_WARPS - 1) / K0_WARPS;
    b4d_launch(k_block_energy, (unsigned)blocks, K0_WARPS * 32, 0, s, u, s21, D, H, W, nvol, zo0, zo1);
}
void b4d_launch_block_energy(const uint16_t *u, uint2 *s21, int D, int H, int W, int nvol, cudaStream_t s) {
    b4d_launch_block_energy_range(u, s21, D, H, W, nvol, 0, D - 3, s);
}

void b4d_launch_match_range(const MatchParams &p, int Ns, int cz0, int cz1, long long tile0, long long tile1,
                            cudaStream_t s) {
    switch (Ns) {
        case 3: launch_ns<3>(p, cz0, cz1, tile0, tile1, s); break;
        case 5: launch_ns<5>(p, cz0, cz1, tile0, tile1, s); break;
        case 7: launch_ns<7>(p, cz0, cz1, tile0, tile1, s); break;
        case 9: launch_ns<9>(p, cz0, cz1, tile0, tile1, s); break;
        case 11: launch_ns<11>(p, cz0, cz1, tile0, tile1, s); break;
        case 13: launch_ns<13>(p, cz0, cz1, tile0, tile1, s); break;
        case 15: launch_ns<15>(p, cz0, cz1, tile0, tile1, s); break;
        default: break;
    }
}
void b4d_launch_match(const MatchParams &p, int Ns, cudaStream_t s) {
    b4d_launch_match_range(p, Ns, 0, (p.g.D + 3) / 4, 0, (long long)p.g.nvol * p.g.tz * p.g.ty * p.g.tx, s);
}
