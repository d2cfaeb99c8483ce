"""Noise level from the MAD of the finest 3-D Haar detail (DESIGN §3.11): the NumPy restatement's properties, the
host-only histogram rule and the argument checks on the CPU; the device kernels bit for bit against the
restatement on the GPU."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("sigma", "mad", "cells")


# ------------------------------------------------- NumPy restatement ----
NOISE_HIST_BINS = 262141  # |d| <= 4 * 65535
NOISE_C = np.sqrt(8.0) * 0.6744897501960817  # std of d under unit white noise, times the normal MAD factor


def _haar_cells(vol):
    """(|d|, data) per 2x2x2 cell at an even origin of one (D, H, W) volume (odd last planes dropped), in plain
    int64: d = sum (-1)^(i+j+k) v[z+i, y+j, x+k]; data = not all 8 voxels are 0 (DESIGN §3.11 items 1-3)."""
    v = np.asarray(vol).astype(np.int64)
    cz, cy, cx = (s // 2 for s in v.shape)
    c = v[: 2 * cz, : 2 * cy, : 2 * cx].reshape(cz, 2, cy, 2, cx, 2)
    d = np.zeros((cz, cy, cx), np.int64)
    nz = np.zeros((cz, cy, cx), bool)
    for i, j, k in np.ndindex(2, 2, 2):
        corner = c[:, i, :, j, :, k]
        d += corner if (i + j + k) % 2 == 0 else -corner
        nz |= corner != 0
    return np.abs(d), nz


def noise_sigma_reference(x, tile=None):
    """DESIGN §3.11 restated: per tile of the C-order grid `tile` (None: one tile per volume), mad = np.median of
    |d| over the tile's data cells, sigma = mad / NOISE_C, cells = their number; NaN for a tile without cells.
    Returns {"sigma", "mad", "cells"} shaped (N,)? + grid, like Denoiser.noise_sigma."""
    x = np.asarray(x)
    vols = x[None] if x.ndim == 3 else x
    D, H, W = vols.shape[1:]
    t = (D + D % 2, H + H % 2, W + W % 2) if tile is None else tuple(int(s) for s in tile)
    grid = tuple(-(-s // ts) for s, ts in zip((D, H, W), t))
    sigma = np.empty((len(vols),) + grid)
    mad = np.empty((len(vols),) + grid)
    cells = np.empty((len(vols),) + grid, np.int64)
    for n, vol in enumerate(vols):
        ad, ok = _haar_cells(vol)
        for iz, iy, ix in np.ndindex(*grid):
            sl = tuple(slice(i * ts // 2, (i + 1) * ts // 2) for i, ts in zip((iz, iy, ix), t))
            vals = ad[sl][ok[sl]]
            cells[n, iz, iy, ix] = vals.size
            mad[n, iz, iy, ix] = np.median(vals) if vals.size else np.nan
            sigma[n, iz, iy, ix] = mad[n, iz, iy, ix] / NOISE_C
    lead = 0 if x.ndim == 3 else slice(None)
    idx = (lead,) + ((0, 0, 0) if tile is None else (Ellipsis,))
    return {"sigma": sigma[idx], "mad": mad[idx], "cells": cells[idx]}


def noise_hist_reference(x):
    """Exact histogram of |d| over every data cell of a volume or batch (262141 bins, int64)."""
    x = np.asarray(x)
    vols = x[None] if x.ndim == 3 else x
    h = np.zeros(NOISE_HIST_BINS, np.int64)
    for vol in vols:
        ad, ok = _haar_cells(vol)
        h += np.bincount(ad[ok], minlength=NOISE_HIST_BINS)
    return h


@pytest.fixture(scope="module")
def lib():
    from b4d import _lib

    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return _lib.load()


@pytest.fixture(scope="module")
def dev():
    import b4d

    return b4d.Denoiser(0)


def _noise(shape, sigma, pedestal, seed):
    rng = np.random.default_rng(seed)
    return np.clip(np.rint(pedestal + sigma * rng.standard_normal(shape)), 0, 65535).astype(np.uint16)


def _same(got, ref):
    for k in KEYS:
        assert np.shape(got[k]) == np.shape(ref[k]), k
        np.testing.assert_array_equal(got[k], ref[k], err_msg=k)


# ---------------------------------------------------------------- CPU ----
def test_noise_header_symbols_are_exported(lib):
    """include/b4d_noise.h is the noise-level part of the C ABI: every function it declares is exported by
    libb4d.so and bound in _lib.NOISE_EXPORTS, and none of them is declared twice."""
    from b4d import _lib

    def declared(name):
        src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", name)).read(), flags=re.S)
        return sorted(set(re.findall(r"\b(b4d_[a-z0-9_]+)\s*\(", src)))

    syms = declared("b4d_noise.h")
    assert syms == sorted(_lib.NOISE_EXPORTS) and not set(syms) & set(declared("b4d.h"))
    for s in syms:
        assert hasattr(lib, s), "libb4d.so does not export %s" % s


def test_restatement_ignores_smooth_backgrounds():
    x = _noise((20, 22, 26), 24.0, 2000.0, 1).astype(np.int64)
    z, y, w = np.meshgrid(*(np.arange(s) for s in x.shape), indexing="ij")
    ad, ok = _haar_cells(x.astype(np.uint16))
    assert ok.all()
    for bg in (np.full(x.shape, 777), 3 * z, 5 * y, 7 * w, y * w, 2 * z + y + 3 * w + y * w):
        ad2, ok2 = _haar_cells((x + bg).astype(np.uint16))
        assert np.array_equal(ad2, ad) and np.array_equal(ok2, ok)


def test_restatement_pure_noise_sigma():
    r = noise_sigma_reference(_noise((128, 128, 128), 24.0, 1000.0, 2))
    assert abs(r["sigma"] / 24.0 - 1.0) < 0.03
    assert r["cells"] == 64 ** 3


@pytest.mark.parametrize("shape", [(6, 6, 6), (6, 6, 8), (9, 7, 11)])
def test_from_hist_equals_restatement(lib, shape):
    import b4d

    x = _noise(shape, 30.0, 500.0, 3)
    h = noise_hist_reference(x)
    r = noise_sigma_reference(x)
    got = b4d.noise_sigma_from_hist(h)
    _same(got, r)
    assert int(h.sum()) == r["cells"]


def test_from_hist_odd_and_even_counts(lib):
    import b4d

    for counts in ({3: 1, 7: 2}, {3: 1, 7: 1}, {0: 2, 600: 1, 900: 1}, {262140: 5}):
        h = np.zeros(NOISE_HIST_BINS, np.int64)
        vals = []
        for v, c in counts.items():
            h[v] = c
            vals += [v] * c
        got = b4d.noise_sigma_from_hist(h)
        mad = np.median(np.array(vals, np.int64))
        assert got["cells"] == len(vals) and got["mad"] == mad
        assert got["sigma"] == mad / (np.sqrt(8.0) * 0.6744897501960817)
    empty = b4d.noise_sigma_from_hist(np.zeros(NOISE_HIST_BINS, np.int64))
    assert empty["cells"] == 0 and np.isnan(empty["sigma"]) and np.isnan(empty["mad"])
    with pytest.raises(ValueError):
        b4d.noise_sigma_from_hist(np.zeros(65536, np.int64))
    bad = np.zeros(NOISE_HIST_BINS, np.int64)
    bad[1] = -1
    with pytest.raises(ValueError):
        b4d.noise_sigma_from_hist(bad)


def test_argument_errors_before_touching_the_device():
    import torch

    import b4d

    ok = np.zeros((8, 8, 8), np.uint16)
    for x, tile in ((ok.astype(np.float32), None), (ok.astype(np.int16), None), (ok[0], None), (ok[None, None], None),
                    (torch.zeros((8, 8, 8), dtype=torch.int32), None), (ok, (4, 4, 3)), (ok, (4, 0, 4)),
                    (ok, (4, -2, 4)), (ok, (4, 4)), (ok, (4, 4, 4, 4))):
        with pytest.raises(ValueError):
            b4d.noise_sigma(x, tile=tile)


# ---------------------------------------------------------------- GPU ----
def _check(dev, x, tile):
    got, hist = dev.noise_sigma(x, tile=tile, return_hist=True)
    _same(got, noise_sigma_reference(x, tile))
    assert hist.dtype == np.int64 and np.array_equal(hist, noise_hist_reference(x))
    return got, hist


def _cells_with(values, shape):
    """A volume whose first len(values) cells hold |d| = values (one non-zero voxel per cell, at its origin); the
    other cells are all zero and skipped."""
    x = np.zeros(shape, np.uint16)
    cz, cy, cx = (s // 2 for s in shape)
    grid = np.zeros(cz * cy * cx, np.uint16)
    grid[: len(values)] = values
    x[: 2 * cz : 2, : 2 * cy : 2, : 2 * cx : 2] = grid.reshape(cz, cy, cx)
    return x


@pytest.mark.gpu
@pytest.mark.parametrize(
    "case",
    ["synth128_t64", "ragged_odd_w", "tile2_12", "whole_volume", "batch5", "batch5_whole", "odd_d_empty_tiles"],
)
def test_device_equals_restatement(dev, case):
    from b4d import synth

    if case == "synth128_t64":
        x, tile = synth.vol(128, 128, 128, seed=0), (64, 64, 64)
    elif case == "ragged_odd_w":
        x, tile = _noise((37, 50, 61), 20.0, 300.0, 4), (16, 8, 32)  # odd W: the 2-byte load path
    elif case == "tile2_12":
        x, tile = _noise((12, 12, 12), 20.0, 300.0, 5), (2, 2, 2)
    elif case == "whole_volume":
        x, tile = synth.vol(72, 80, 96, seed=1), None
    elif case == "batch5":
        x, tile = _noise((5, 40, 40, 40), 15.0, 100.0, 6), (16, 16, 16)
    elif case == "batch5_whole":
        x, tile = _noise((5, 40, 40, 40), 15.0, 100.0, 7), None
    else:  # D = 37 with tz = 36: the second tile layer holds plane 36 only, no cell, NaN
        x, tile = _noise((37, 20, 24), 20.0, 300.0, 8), (36, 8, 8)
    got, _ = _check(dev, x, tile)
    if case == "odd_d_empty_tiles":
        assert np.all(got["cells"][1] == 0) and np.all(np.isnan(got["sigma"][1]))


@pytest.mark.gpu
def test_device_extremes(dev):
    z, y, w = np.meshgrid(np.arange(16), np.arange(18), np.arange(20), indexing="ij")
    board = (65535 * ((z + y + w) % 2)).astype(np.uint16)
    got, hist = _check(dev, board, (8, 8, 8))
    assert np.all(got["mad"] == 262140.0) and hist[262140] == 8 * 9 * 10
    got, _ = _check(dev, np.full((16, 16, 16), 500, np.uint16), (8, 8, 8))
    assert np.all(got["sigma"] == 0.0) and np.all(got["cells"] == 64)
    got, _ = _check(dev, np.zeros((8, 8, 8), np.uint16), None)
    assert got["cells"] == 0 and np.isnan(got["sigma"])
    half = _noise((32, 32, 32), 24.0, 400.0, 9)
    half[:, :, :16] = 0  # zero-filled padding: its cells are skipped
    got, _ = _check(dev, half, (16, 16, 16))
    assert np.all(got["cells"][:, :, 0] == 0) and np.all(got["cells"][:, :, 1] == 512)
    # the two middle ranks in different high-digit bins (|d| >> 9 = 0 and 1), and inside them not at the bin edges
    rng = np.random.default_rng(10)
    vals = np.concatenate([rng.integers(1, 512, 32), rng.integers(512, 1100, 32)]).astype(np.uint16)
    rng.shuffle(vals)
    x = _cells_with(vals, (8, 8, 16))
    got, _ = _check(dev, x, None)
    s = np.sort(vals.astype(np.int64))
    assert (s[31] >> 9, s[32] >> 9) == (0, 1) and got["mad"] == (s[31] + s[32]) / 2


@pytest.mark.gpu
def test_slab_histograms_sum_to_the_volume(dev):
    import b4d
    from b4d import synth

    x = synth.vol(60, 48, 40, seed=2)
    whole, hist = dev.noise_sigma(x, return_hist=True)
    parts = [dev.noise_sigma(x[a:b], return_hist=True)[1] for a, b in ((0, 20), (20, 42), (42, 60))]
    total = np.sum(parts, axis=0)
    assert np.array_equal(total, hist)
    _same(b4d.noise_sigma_from_hist(total), whole)


@pytest.mark.gpu
def test_torch_cuda_input(dev):
    import torch

    import b4d

    x = _noise((2, 24, 30, 34), 24.0, 300.0, 11)
    ref = dev.noise_sigma(x, tile=(8, 10, 12))
    _same(dev.noise_sigma(torch.from_numpy(x.view(np.int16)).view(torch.uint16).cuda(), tile=(8, 10, 12)), ref)
    # a device view 2 bytes past an allocation: not 4-byte aligned, the 2-byte load path with even W
    flat = torch.zeros(x.size + 1, dtype=torch.int16, device="cuda")
    flat[1:] = torch.from_numpy(x.view(np.int16).reshape(-1)).cuda()
    view = flat[1:].view(torch.uint16).view(x.shape)
    assert view.data_ptr() % 4 == 2
    _same(b4d.noise_sigma(view, tile=(8, 10, 12)), ref)


@pytest.mark.gpu
def test_device_512_cubed(dev):
    from b4d import synth

    x = synth.vol(512, 512, 512, seed=4)
    got = dev.noise_sigma(x, tile=(64, 64, 64))
    _same(got, noise_sigma_reference(x, (64, 64, 64)))
    assert got["sigma"].shape == (8, 8, 8)


def _motivation_tile(kind, seed=1):
    """One 64^3 tile of the synth clean field on a pedestal of 200 plus white noise of sigma 24, with a z ramp of 2
    counts per plane and / or a smooth texture (white noise blurred with sigma 6 voxels, std 50)."""
    from scipy import ndimage

    from b4d import synth

    rng = np.random.default_rng(seed)
    clean = synth.clean_tile(seed)[:64, :64, :64].astype(np.float64) + (200.0 - synth.PEDESTAL)
    if "ramp" in kind:
        clean = clean + 2.0 * np.arange(64.0)[:, None, None]
    if "texture" in kind:
        f = ndimage.gaussian_filter(rng.standard_normal((64, 64, 64)), 6.0, mode="wrap")
        clean = clean + f * (50.0 / f.std())
    return np.clip(np.rint(clean + 24.0 * rng.standard_normal(clean.shape)), 0, 65535).astype(np.uint16)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["ramp", "texture", "texture+ramp"])
def test_sigma_of_textured_background(dev, kind):
    x = _motivation_tile(kind)
    got = dev.noise_sigma(x)
    assert abs(got["sigma"] / 24.0 - 1.0) < 0.05
    # the intensity statistic counts the background as noise: the reason this estimator exists
    assert dev.tile_stats(x)["sigma"] > 2 * 24.0
