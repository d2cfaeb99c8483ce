"""The block matcher's selection schedule and acceptance limits (csrc/b4d_match.cu, DESIGN.md §4 and §5).

`k_match` keeps, per reference block, only the keys at or below a running bound in a 512-entry survivor list.  On
common data the list never fills; when it does, the reference runs again with the final bound (mode 1, counted in
`retry_refs`) and, if that overflows too, takes K rounds of "smallest key above the previous one" (mode 2,
`slow_refs`).  In the byte kernel a reference PAIR whose list overflows goes back to the one-reference loop.

`schedule` restates in NumPy what one warp does for one reference, so that it predicts both counters exactly.  The
generators below build volumes whose windows make the schedule overflow: constant along x (every candidate of a
window row ties in SSD, so keys arrive in index order) and a (z, y) pattern found by a seeded hill climb on the
model.  The GPU tests check the match lists against the oracle's brute force, the counters against the model and
the TMA staging against its fallback, on byte, narrow and wide tiles.  The acceptance-limit tests place SSDs and
tile ranges exactly at the thresholds of the kernel arithmetic.

Which windows can overflow at all: in one iteration a key at or below the bound lies in one of the K lanes with the
smallest running minimum (K = 32: 16 lanes by the second minimum, plus at most one key in each other lane), so mode 0
keeps at most ITERS * min(K, 16) * Ns (+ 16 ITERS for K = 32) keys, and mode 1 at most min(K, 16) * ITERS * Ns (+ 16).
That is <= 512 for every K at Ns = 9 and for K <= 8 at Ns = 11: only Ns >= 11 (and Ns >= 13 for K = 8) can
reach these paths.
"""
import functools
import math
import os

import numpy as np
import pytest

CAP = 512
INVALID = 0xFFFFFFFF
TAU_HT = 2.9527
SHAPE = (36, 36, 40)  # W % 8 == 0: the byte kernel stages through TMA unless B4D_NO_TMA is set
TARGET = (12, 12)  # (oz, oy) of the references that see the generated pattern: the first layer of tile (1, 1)


def ref_origins(n):
    o = list(range(0, n - 3, 3))
    if (n - 4) % 3:
        o.append(n - 4)
    return np.array(o)


def kb_of(ns):
    return 11 if ns ** 3 <= 2048 else 12


def tau_int(tau, sigma):
    """tau_for / tau_int: floor(tau * sigma^2 * 64) from float32 arguments, evaluated in double."""
    s = float(np.float32(sigma))
    return math.floor(float(np.float32(tau)) * s * s * 64.0)


def unit_order(ns):
    """Geo<NS>::order_at: the 32-unit groups of the window, centre-out."""
    units = ns * ns
    iters = (units + 31) // 32
    mc = (units // 2) // 32
    out = []
    for k in range(2 * iters + 2):
        off = (k + 1) // 2
        m = mc + off if k & 1 else mc - off
        if 0 <= m < iters:
            out.append(m)
    return out


# ------------------------------------------------------------------ the host model ------
def window_ssd(vol, ns):
    """Exact SSD of every reference block to every candidate of its Ns^3 window: int64 [R, Ns^3] in window-index
    order (dz * Ns + dy) * Ns + dx, -1 where the candidate leaves the volume."""
    v = vol.astype(np.int64)
    D, H, W = v.shape
    r = ns // 2
    rz, ry, rx = ref_origins(D), ref_origins(H), ref_origins(W)
    vp = np.zeros((D + 2 * r, H + 2 * r, W + 2 * r), np.int64)
    vp[r:r + D, r:r + H, r:r + W] = v
    out = np.empty((len(rz), len(ry), len(rx), ns, ns, ns), np.int64)
    ok = [[(o + d >= 0) & (o + d <= n - 4) for d in range(-r, r + 1)] for o, n in ((rz, D), (ry, H), (rx, W))]
    for a in range(ns):
        for b in range(ns):
            for c in range(ns):
                d2 = (vp[a:a + D, b:b + H, c:c + W] - v) ** 2
                s = d2[:, :, rx] + d2[:, :, rx + 1] + d2[:, :, rx + 2] + d2[:, :, rx + 3]
                s = s[:, ry] + s[:, ry + 1] + s[:, ry + 2] + s[:, ry + 3]
                s = s[rz] + s[rz + 1] + s[rz + 2] + s[rz + 3]
                valid = ok[0][a][:, None, None] & ok[1][b][None, :, None] & ok[2][c][None, None, :]
                out[:, :, :, a, b, c] = np.where(valid, s, -1)
    return out.reshape(-1, ns ** 3)


def window_keys(ssd, ns, tau):
    """key = SSD << KB | window index for accepted candidates (0 <= SSD <= tau), INVALID otherwise."""
    idx = np.arange(ns ** 3, dtype=np.int64)
    return np.where((ssd >= 0) & (ssd <= tau), (ssd << kb_of(ns)) | idx, INVALID)


def schedule(keys, ns, K, tau):
    """One warp per reference (k_match, one-reference loop): per-lane running minimum (second minimum for K = 32)
    over the units visited centre-out, bound B refined by the K-th smallest of them before each take test.
    Returns (mode-0 survivor count, final bound, keys <= final bound) per reference."""
    R = keys.shape[0]
    kb = kb_of(ns)
    dmax = (1 << (32 - kb)) - 1
    keymax = (min(tau, dmax - 1) << kb) | ((1 << kb) - 1)
    units = ns * ns
    rows = np.full((R, ((units + 31) // 32) * 32, ns), INVALID, np.int64)
    rows[:, :units] = keys.reshape(R, units, ns)
    l1 = np.full((R, 32), INVALID, np.int64)
    l2 = l1.copy()
    B = np.full(R, keymax, np.int64)
    n0 = np.zeros(R, np.int64)
    k32 = K == 32
    kth = 15 if k32 else K - 1
    for m in unit_order(ns):
        blk = rows[:, m * 32:(m + 1) * 32]  # lane l holds unit 32 m + l, its Ns keys along dx
        for j in range(ns):
            if k32:
                l2 = np.minimum(l2, np.maximum(l1, blk[:, :, j]))
            l1 = np.minimum(l1, blk[:, :, j])
        B = np.minimum(B, np.partition(l2 if k32 else l1, kth, axis=1)[:, kth])
        n0 += (blk <= B[:, None, None]).sum((1, 2))
    return n0, B, (keys <= B[:, None]).sum(1)


def predicted_stats(keys, ns, K, tau):
    n0, _, n1 = schedule(keys, ns, K, tau)
    return {"retry_refs": int((n0 > CAP).sum()), "slow_refs": int(((n0 > CAP) & (n1 > CAP)).sum())}


def complete_selection(keys, ns, K, tau, shape):
    """The model's match lists in the form of match_stage1: modes 0 and 1 rank-sort the keys <= the final bound,
    mode 2 takes the K smallest accepted keys; K' = the largest power of two <= min(K, found)."""
    n0, B, n1 = schedule(keys, ns, K, tau)
    slow = (n0 > CAP) & (n1 > CAP)
    cut = np.where(slow, INVALID - 1, B)
    srt = np.sort(np.where(keys <= cut[:, None], keys, INVALID), 1)[:, :K]
    found = (srt != INVALID).sum(1)
    cnt = np.where(found > 0, 1 << np.floor(np.log2(np.maximum(found, 1))).astype(np.int64), 0)
    D, H, W = shape
    r = ns // 2
    rz, ry, rx = ref_origins(D), ref_origins(H), ref_origins(W)
    oz, oy, ox = (a.ravel() for a in np.meshgrid(rz, ry, rx, indexing="ij"))
    wi = srt & ((1 << kb_of(ns)) - 1)
    cz, cy, cx = oz[:, None] - r + wi // (ns * ns), oy[:, None] - r + (wi // ns) % ns, ox[:, None] - r + wi % ns
    take = np.arange(K)[None, :] < cnt[:, None]
    idx = np.where(take, (cz * (H - 3) + cy) * (W - 3) + cx, -1).astype(np.int32)
    ssd = np.where(take, srt >> kb_of(ns), -1).astype(np.int64).astype(np.uint64)
    return idx, ssd, cnt.astype(np.int32)


def tile_classes(vol, ns):
    """k_tile_class: exact range of every matcher tile's staged neighbourhood -> (byte tiles, wide tiles, classes)."""
    r, E = ns // 2, ns + 12
    orig = [ref_origins(n) for n in vol.shape]
    cls = {}
    for tz in range(0, len(orig[0]), 4):
        for ty in range(0, len(orig[1]), 4):
            for tx in range(0, len(orig[2]), 4):
                b = [orig[0][tz] - r, orig[1][ty] - r, orig[2][tx] - r]
                nb = vol[max(b[0], 0):b[0] + E, max(b[1], 0):b[1] + E, max(b[2], 0):b[2] + E].astype(np.int64)
                rng = int(nb.max() - nb.min())
                cls[(tz // 4, ty // 4, tx // 4)] = "byte" if rng <= 255 else ("narrow" if rng <= 8191 else "wide")
    v = list(cls.values())
    return v.count("byte"), v.count("wide"), cls


# ------------------------------------------------------------------ generators -----------
def pattern_ssd(p, ns):
    """SSD [P, Ns, Ns] of the centre block of (Ns + 3)^2 (z, y) patterns, constant along x, to each window row."""
    r = ns // 2
    ref = p[:, r:r + 4, r:r + 4]
    s = np.empty((p.shape[0], ns, ns), np.int64)
    for a in range(ns):
        for b in range(ns):
            s[:, a, b] = 4 * ((p[:, a:a + 4, b:b + 4] - ref) ** 2).sum((1, 2))
    return s


@functools.lru_cache(maxsize=None)
def overflow_pattern(ns, path, ks, seed=1, pop=128, rounds=150):
    """Seeded hill climb for an (Ns + 3)^2 pattern of values < 120 that maximises, over the K in `ks`, the smallest
    mode-0 survivor count (path "retry") or count of keys under the final bound (path "slow") of the centre
    reference at sigma = 24."""
    rng = np.random.default_rng(seed)
    tau = tau_int(TAU_HT, 24.0)
    which = 0 if path == "retry" else 2
    idx = np.arange(ns ** 3).reshape(ns, ns, ns)

    def score(p):
        s = np.broadcast_to(pattern_ssd(p, ns)[:, :, :, None], (p.shape[0], ns, ns, ns))
        keys = np.where(s <= tau, (s << kb_of(ns)) | idx, INVALID).reshape(p.shape[0], -1)
        return np.min([schedule(keys, ns, K, tau)[which] for K in ks], 0)

    cand = rng.integers(0, 120, (pop, ns + 3, ns + 3))
    sc = score(cand)
    best, bs = cand[np.argmax(sc)], sc.max()
    for _ in range(rounds):
        cand = np.repeat(best[None], pop, 0)
        pos = rng.integers(0, ns + 3, (pop, 2))
        cand[np.arange(pop), pos[:, 0], pos[:, 1]] = rng.integers(0, 120, pop)
        sc = score(cand)
        if sc.max() >= bs:
            best, bs = cand[np.argmax(sc)], sc.max()
    return best


def search_ks(ns, path, K):
    """The K set a case's pattern is searched for: K = 8 has its own pattern where it can overflow (retry at
    Ns = 15); every other case uses the pattern found for K = 16 and 32."""
    return (8,) if (K == 8 and ns == 15 and path == "retry") else (16, 32)


@functools.lru_cache(maxsize=None)
def overflow_case(ns, path, ks, tile):
    """(volume, sigma) of a generated case.  The pattern sits in the (z, y) window of the TARGET references, edge
    values continue outside it, the volume is constant along x.  tile = "byte": as generated; "narrow": pattern
    and sigma scaled by 3 (range > 255, same key order); "wide": one voxel of 65535 in the staged neighbourhood of
    the TARGET tile, outside the windows of the TARGET references."""
    p = overflow_pattern(ns, path, ks).astype(np.int64)
    r = ns // 2
    D, H, W = SHAPE
    z0, y0 = TARGET[0] - r, TARGET[1] - r
    plane = np.pad(p, ((z0, D - z0 - ns - 3), (y0, H - y0 - ns - 3)), mode="edge")
    vol = np.broadcast_to(plane[:, :, None], SHAPE).copy()
    sigma = 24.0
    if tile == "narrow":
        vol *= 3
        sigma = 72.0
    if tile == "wide":
        vol[TARGET[0] + r + 12, TARGET[1], 20] = 65535  # last plane of the tile's neighbourhood
    return vol.astype(np.uint16), sigma


@functools.lru_cache(maxsize=None)
def overflow_ssd(ns, path, ks, tile):
    vol, _ = overflow_case(ns, path, ks, tile)
    return window_ssd(vol, ns)


def target_rows(ns):
    """Reference indices of the TARGET references whose x window is complete."""
    D, H, W = SHAPE
    rz, ry, rx = ref_origins(D), ref_origins(H), ref_origins(W)
    iz, iy = int(np.flatnonzero(rz == TARGET[0])[0]), int(np.flatnonzero(ry == TARGET[1])[0])
    ix = np.flatnonzero((rx >= ns // 2) & (rx <= W - 4 - ns // 2))
    return (iz * len(ry) + iy) * len(rx) + ix


# Generated cases whose targeted path the model shows reached (the others run for parity and counters only)
REACHED = {("retry", ns, K) for ns in (11, 13, 15) for K in (16, 32)} | {("retry", 15, 8)}
REACHED |= {("slow", ns, K) for ns in (11, 13, 15) for K in (16, 32)}
GEN_CASES = [(path, ns, K, tile) for path in ("retry", "slow") for ns in (9, 11, 13, 15) for K in (8, 16, 32)
             for tile in ("byte", "narrow", "wide")]


def case_prediction(path, ns, K, tile):
    ks = search_ks(ns, path, K)
    vol, sigma = overflow_case(ns, path, ks, tile)
    tau = tau_int(TAU_HT, sigma)
    keys = window_keys(overflow_ssd(ns, path, ks, tile), ns, tau)
    return vol, sigma, tau, keys


# ------------------------------------------------------------------ CPU tests -----------
def test_unit_order_matches_the_kernel_table():
    # Geo<NS>::ORDER for the windows that can overflow (centre group first, then alternately above and below)
    assert unit_order(11) == [1, 2, 0, 3]
    assert unit_order(13) == [2, 3, 1, 4, 0, 5]
    assert unit_order(15) == [3, 4, 2, 5, 1, 6, 0, 7]
    assert unit_order(9) == [1, 2, 0]


@pytest.mark.parametrize("path,ns,K", sorted(REACHED))
@pytest.mark.parametrize("tile", ["byte", "narrow", "wide"])
def test_generators_reach_their_path_in_the_model(path, ns, K, tile):
    _, _, tau, keys = case_prediction(path, ns, K, tile)
    n0, _, n1 = schedule(keys, ns, K, tau)
    rows = target_rows(ns)
    assert (n0[rows] > CAP).all(), (path, ns, K, tile, n0[rows])
    if path == "slow":
        assert (n1[rows] > CAP).all(), (path, ns, K, tile, n1[rows])
    st = predicted_stats(keys, ns, K, tau)
    assert st["retry_refs"] >= len(rows) and (path == "retry" or st["slow_refs"] >= len(rows))
    vol, _ = overflow_case(ns, path, search_ks(ns, path, K), tile)
    nbyte, nwide, cls = tile_classes(vol, ns)
    assert cls[(1, 1, 1)] == tile  # the TARGET references' tile


@pytest.mark.parametrize("ns,K", [(9, 8), (9, 16), (9, 32), (11, 8)])
def test_windows_that_cannot_overflow(ns, K):
    """The reachability bound of the module docstring, and the generators' best effort staying under it."""
    iters = (ns * ns + 31) // 32
    lanes = min(K, 16)
    assert iters * (lanes * ns + (16 if K == 32 else 0)) <= CAP
    for path in ("retry", "slow"):
        _, _, tau, keys = case_prediction(path, ns, K, "byte")
        assert predicted_stats(keys, ns, K, tau) == {"retry_refs": 0, "slow_refs": 0}


@pytest.mark.parametrize("path,ns,K", [("retry", 11, 16), ("slow", 11, 32), ("retry", 15, 8), ("slow", 13, 16)])
def test_model_selects_what_the_oracle_selects(path, ns, K, oracle_lib):
    vol, sigma, tau, keys = case_prediction(path, ns, K, "byte")
    mi, ms, mc = complete_selection(keys, ns, K, tau, vol.shape)
    oi, os_, oc = oracle_lib.Oracle("f64", search_ht=ns, k_ht=K).match_stage1(vol, sigma)
    assert np.array_equal(mc, oc) and np.array_equal(mi, oi) and np.array_equal(ms, os_)


@pytest.mark.parametrize("seed,ns,K", [(3, 11, 16), (5, 13, 32), (8, 15, 8)])
def test_model_selects_what_the_oracle_selects_on_synthetic_volumes(seed, ns, K, oracle_lib):
    from b4d import synth

    vol = synth.vol(22, 21, 24, seed=seed)
    tau = tau_int(TAU_HT, 24.0)
    keys = window_keys(window_ssd(vol, ns), ns, tau)
    mi, ms, mc = complete_selection(keys, ns, K, tau, vol.shape)
    oi, os_, oc = oracle_lib.Oracle("f64", search_ht=ns, k_ht=K).match_stage1(vol, 24.0)
    assert np.array_equal(mc, oc) and np.array_equal(mi, oi) and np.array_equal(ms, os_)
    assert predicted_stats(keys, ns, K, tau) == {"retry_refs": 0, "slow_refs": 0}


# ------------------------------------------------------------------ acceptance-limit volumes ---
def sigma_for_tau(target, tau=1.0):
    """A float32 sigma whose tau_for(tau, sigma) is exactly `target`."""
    s = np.float32(math.sqrt(target / 64.0 / tau))
    for _ in range(64):
        v = tau_int(tau, s)
        if v == target:
            return float(s)
        s = np.nextafter(s, np.float32(np.inf if v < target else 0), dtype=np.float32)
    raise AssertionError("no float32 sigma gives tau %d" % target)


def split_volume(shape, lo, delta):
    """Two flat regions along x: lo for x < W/2, lo + delta above."""
    vol = np.full(shape, lo, np.int64)
    vol[:, :, shape[2] // 2:] += delta
    return vol.astype(np.uint16)


def stamp_values(total):
    """64 offsets in [0, 255] whose squares sum to `total`."""
    q = math.isqrt(total // 64)
    for k in range(62):  # k voxels at q - 1, 61 - k at q, three free
        rest = total - k * (q - 1) ** 2 - (61 - k) * q * q
        for a in range(min(255, math.isqrt(max(rest, 0))), -1, -1):
            for b in range(min(a, math.isqrt(rest - a * a)), -1, -1):
                c = math.isqrt(rest - a * a - b * b)
                if c * c == rest - a * a - b * b and c <= b:
                    return np.array([q - 1] * k + [q] * (61 - k) + [a, b, c], np.int64)
    raise AssertionError(total)


ISO_SHAPE = (30, 30, 40)
# Reference cubes (oz, oy, ox).  oz = 6: cube A, oz = 21: cube B.  On byte tiles ox = 18 / 21 are the two members of
# an interior pair (saturating key path min(SSD, DMAX)), ox = 0 / 3 the two members of an x-edge pair (the tested
# paths `da <= tau`, `db <= tau`), ox = 36 sits in a tile with a flush origin, matched by the one-reference loop.
ISO_CUBES = [(oz, oy, ox) for oz in (6, 21) for oy, ox in ((6, 18), (6, 0), (6, 36), (21, 21), (21, 3))]


def isolated_volume(ns, tau, tile):
    """References whose group size changes with the acceptance of SSD = tau.  Flat cubes of value v (v^2 > tau) in
    a zero background, so that every candidate holding a background voxel is above tau and no cube lies in another
    cube's window; stamp blocks 5 voxels away (a background plane between) differ from their cube by exactly the
    listed SSDs.  Cube A accepts itself, tau / 2, 3 tau / 4 and tau: K' = 4, and 2 if tau were rejected.  Cube B
    accepts itself, tau / 2 and 3 tau / 4 but not tau + 1: K' = 2, and 4 if tau + 1 were accepted.  v = 200 keeps the
    tiles byte tiles for an ordinary tau; tau at the key ceiling needs v = 3000 (narrow tiles).  tile = "narrow" /
    "wide" adds voxels of 400 / 65535 to the background of every cube's tile (a candidate holding one is rejected
    anyway)."""
    v = 200 if tau < 40000 else 3000
    vol = np.zeros(ISO_SHAPE, np.int64)
    for oz, oy, ox in ISO_CUBES:
        top = tau if oz == 6 else tau + 1
        vol[oz:oz + 4, oy:oy + 4, ox:ox + 4] = v
        for (dz, dy), t in zip(((5, 0), (0, 5), (-5, 0)), (top, tau - tau // 4, tau - tau // 2)):
            z, y = oz + dz, oy + dy
            vol[z:z + 4, y:y + 4, ox:ox + 4] = v - stamp_values(t).reshape(4, 4, 4)
    fill = {"byte": 0, "narrow": 400, "wide": 65535}[tile]
    if fill:
        vol[15, 15, 15] = vol[15, 15, 33] = fill
    return vol.astype(np.uint16), sigma_for_tau(tau)


def isolated_refs():
    """{(oz, oy, ox): reference index} of the cube references of isolated_volume."""
    rz, ry, rx = (list(ref_origins(n)) for n in ISO_SHAPE)
    return {c: (rz.index(c[0]) * len(ry) + ry.index(c[1])) * len(rx) + rx.index(c[2]) for c in ISO_CUBES}


def iso_expected(c, tau):
    """(K', SSDs of the list) of cube reference c."""
    return (4, [0, tau - tau // 2, tau - tau // 4, tau]) if c[0] == 6 else (2, [0, tau - tau // 2])


ORDINARY_TAU = 30000
ISO_CASES = [(ns, tau, tile) for ns in (11, 13) for tau, tiles in
             ((ORDINARY_TAU, ("byte", "narrow", "wide")), ((1 << (32 - kb_of(ns))) - 2, ("narrow", "wide")))
             for tile in tiles]


@pytest.mark.parametrize("ns,tau,tile", ISO_CASES)
def test_acceptance_volumes_are_what_they_claim(ns, tau, tile):
    """In the model, each cube reference's group size depends on the decision at the threshold: it changes if the
    stamp at tau (A) were rejected or the one at tau + 1 (B) accepted."""
    vol, sigma = isolated_volume(ns, tau, tile)
    assert tau_int(1.0, sigma) == tau
    ssd = window_ssd(vol, ns)
    _, lssd, lcnt = complete_selection(window_keys(ssd, ns, tau), ns, 16, tau, vol.shape)
    for c, ri in isolated_refs().items():
        cnt, want = iso_expected(c, tau)
        assert lcnt[ri] == cnt and list(lssd[ri, :cnt]) == want
        # the other decision at the threshold (counted on the SSDs: at the ceiling tau + 1 does not fit the key)
        other = tau - 1 if c[0] == 6 else tau + 1
        n = int(((ssd[ri] >= 0) & (ssd[ri] <= other)).sum())
        assert 1 << (n.bit_length() - 1) != cnt
    _, _, cls = tile_classes(vol, ns)
    rz, ry, rx = (list(ref_origins(n)) for n in ISO_SHAPE)
    assert {cls[(rz.index(c[0]) // 4, ry.index(c[1]) // 4, rx.index(c[2]) // 4)] for c in ISO_CUBES} == {tile}


def test_threshold_arithmetic():
    lim11, lim12 = (1 << 21) - 2, (1 << 20) - 2
    assert tau_int(1.0, sigma_for_tau(lim11)) == lim11 and tau_int(1.0, sigma_for_tau(lim12)) == lim12
    assert 64 * 8192 ** 2 == 1 << 32 and 64 * 8191 ** 2 < 1 << 32


# ------------------------------------------------------------------ GPU tests -----------
@pytest.fixture(scope="module")
def b4d_mod():
    import b4d

    return b4d


def _denoiser(b4d_mod, ns, K, tau=TAU_HT, stages=2):
    prof = b4d_mod.BM4DProfile(search_window_ht=(ns // 2,) * 3, max_stack_size_ht=K, tau_match_ht=tau)
    return b4d_mod.Denoiser(0, prof, stages)


def _match_and_compare(d, oracle_lib, vol, sigma, ns, K, tau_match=TAU_HT):
    gi, gs, gc = d.match_stage1(vol, sigma)
    stats = d.last_match_stats()
    oi, os_, oc = oracle_lib.Oracle("f64", search_ht=ns, k_ht=K, tau_ht=tau_match).match_stage1(vol, sigma)
    assert np.array_equal(gc, oc), "count differs at %d references" % int((gc != oc).sum())
    assert np.array_equal(gi, oi), "idx differs at %d references" % int((gi != oi).any(1).sum())
    assert np.array_equal(gs, os_)
    os.environ["B4D_NO_TMA"] = "1"
    try:
        ti, ts, tc = d.match_stage1(vol, sigma)
        tstats = d.last_match_stats()
    finally:
        del os.environ["B4D_NO_TMA"]
    assert np.array_equal(ti, gi) and np.array_equal(ts, gs) and np.array_equal(tc, gc)
    assert tstats == stats
    return stats, (gi, gs, gc)


def _expected_stats(vol, ns, K, tau, keys=None):
    if keys is None:
        keys = window_keys(window_ssd(vol, ns), ns, tau)
    nbyte, nwide, _ = tile_classes(vol, ns)
    return dict(predicted_stats(keys, ns, K, tau), byte_tiles=nbyte, wide_tiles=nwide)


@pytest.mark.gpu
@pytest.mark.parametrize("path,ns,K,tile", GEN_CASES)
def test_overflow_paths_equal_the_oracle_and_the_model(path, ns, K, tile, b4d_mod, oracle_lib):
    vol, sigma, tau, keys = case_prediction(path, ns, K, tile)
    d = _denoiser(b4d_mod, ns, K)
    try:
        stats, _ = _match_and_compare(d, oracle_lib, vol, sigma, ns, K)
    finally:
        d.close()
    want = _expected_stats(vol, ns, K, tau, keys)
    print("[%s Ns=%d K=%d %s] gpu %s model %s" % (path, ns, K, tile, stats, want))
    assert stats == want
    if (path, ns, K) in REACHED:
        assert stats["retry_refs"] > 0 and (path == "retry" or stats["slow_refs"] > 0)
    assert (stats["byte_tiles"] > 0) if tile == "byte" else True
    assert (stats["wide_tiles"] > 0) == (tile == "wide")


def _stage2_image(basic, vol):
    """The stage-2 matching image of a uint16 input: clamp(rint(basic) + centre shift, 0, 65535)."""
    lo, hi = float(vol.min()), float(vol.max())
    shift = int(math.floor((65535.0 - (hi - lo)) * 0.5) - lo)
    return np.clip(np.rint(basic).astype(np.int64) + shift, 0, 65535).astype(np.uint16)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["retry", "slow"])
@pytest.mark.parametrize("tile", ["byte", "narrow", "wide"])
def test_overflow_paths_denoise_bit_exact_vs_mirror(path, tile, b4d_mod, oracle_lib):
    """Default profile (Ns = 11, K = 16 / 32): both stages equal the float32 mirror bit for bit, the fixed-point
    accumulators integer for integer.  last_match_stats after a two-stage call is the SUM of both matchers: stage 1
    resets the counters, the stage-2 front end adds to them."""
    vol, sigma, tau, keys = case_prediction(path, 11, 16, tile)
    st1 = _expected_stats(vol, 11, 16, tau, keys)
    assert st1["retry_refs"] > 0 and (path == "retry" or st1["slow_refs"] > 0)
    d = b4d_mod.Denoiser(0)
    try:
        for stages in (1, 2):
            d.set_profile(b4d_mod.BM4DProfile(), stages)
            y = d.denoise(vol, sigma)
            stats = d.last_match_stats()
            gn, gw = d.debug_accumulators(vol.size)
            o = oracle_lib.Oracle("mirror", stages=stages)
            m = o.denoise(vol, sigma)
            on, ow = o.accumulators(vol.size)
            assert np.array_equal(y, m), "stage %d: max-abs %g" % (stages, np.abs(y - m).max())
            assert np.array_equal(gn, on) and np.array_equal(gw, ow), "stage %d accumulators" % stages
            if stages == 1:
                basic = y
                assert stats == st1
            else:
                u2 = _stage2_image(basic, vol)
                st2 = _expected_stats(u2, 11, 32, tau_int(0.7693, sigma))
                assert stats == {k: st1[k] + st2[k] for k in st1}, (stats, st1, st2)
    finally:
        d.close()


@pytest.mark.gpu
@pytest.mark.parametrize("delta", [8191, 8192, 255, 256])
def test_tile_range_limits(delta, b4d_mod, oracle_lib):
    """Two flat regions delta apart.  8192: the tile is wide and the cross SSD 64 * 8192^2 = 2^32 (0 modulo 2^32)
    is rejected; 8191: narrow, 64 * 8191^2 < 2^32 exact.  255 / 256: the tile is classified byte / general, and the
    byte window holds offsets up to 255."""
    vol = split_volume((20, 22, 32), 700, delta)
    d = _denoiser(b4d_mod, 11, 16)
    try:
        stats, _ = _match_and_compare(d, oracle_lib, vol, 24.0, 11, 16)
    finally:
        d.close()
    assert stats == _expected_stats(vol, 11, 16, tau_int(TAU_HT, 24.0))
    assert (stats["wide_tiles"] > 0) == (delta == 8192)
    nb = tile_classes(vol, 11)[0]
    assert (nb == len(tile_classes(vol, 11)[2])) == (delta <= 255)


@pytest.mark.gpu
@pytest.mark.parametrize("ns,tau,tile", ISO_CASES)
def test_ssd_equal_to_tau_is_accepted(ns, tau, tile, b4d_mod, oracle_lib):
    """SSD = tau is accepted and tau + 1 rejected, on byte, narrow and wide tiles at an ordinary tau and at the key
    ceiling 2^(32 - KB) - 2 (where tau + 1 = DMAX, the value the saturating key path clamps to): in both members of
    an interior and of an x-edge byte pair, in the one-reference byte loop and in the general kernel."""
    vol, sigma = isolated_volume(ns, tau, tile)
    K = 16
    d = _denoiser(b4d_mod, ns, K, tau=1.0)
    try:
        stats, (gi, gs, gc) = _match_and_compare(d, oracle_lib, vol, sigma, ns, K, 1.0)
    finally:
        d.close()
    assert stats == _expected_stats(vol, ns, K, tau)
    for c, ri in isolated_refs().items():
        cnt, want = iso_expected(c, tau)
        assert gc[ri] == cnt and list(gs[ri, :cnt]) == want, c


@pytest.mark.gpu
@pytest.mark.parametrize("other", [65435, 62535, 0])
def test_reference_blocks_at_full_scale(other, b4d_mod, oracle_lib):
    """Blocks of 65535: S2 = 64 * 65535^2 needs the 6 high bits packed beside S1.  Regions at 65535 and 65435
    (SSD 640 000 = tau at sigma 100, tau 1.0), plus planes at `other`: byte (65435), narrow (62535) or wide (0)."""
    vol = split_volume((20, 22, 32), 65435, 100).astype(np.int64)
    vol[:, :, :8] = 65535
    vol[15:, :, :] = other
    vol = vol.astype(np.uint16)
    d = _denoiser(b4d_mod, 11, 16, tau=1.0)
    try:
        stats, _ = _match_and_compare(d, oracle_lib, vol, 100.0, 11, 16, 1.0)
    finally:
        d.close()
    assert stats == _expected_stats(vol, 11, 16, 640000)
    assert (stats["wide_tiles"] > 0) == (other == 0)
