"""Poisson-Gaussian noise (DESIGN §3.12): the noise-level function (NLF), the generalized Anscombe transform (GAT)
and denoising through it.  The NumPy restatement of the contract (int64 cells, float64 arithmetic in the
contract's order) and its properties on the CPU; the device kernels bit for bit against it on the GPU."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ------------------------------------------------- NumPy restatement ----
NOISE_C = np.sqrt(8.0) * 0.6744897501960817  # as DESIGN §3.11
S15 = np.sqrt(1.5)
C1 = 0.25 * S15
C2 = 0.625 * S15


def default_edges():
    return np.array([0.0] + [32.0 * 2.0 ** (k / 3.0) for k in range(34)])


def _cells(vol):
    """(|d|, s) of the data cells (s > 0) of one volume: d the unnormalised HHH Haar detail, s the sum of the 8
    voxels, both int64 (DESIGN §3.11 items 1-3, §3.12)."""
    v = np.asarray(vol).astype(np.int64)
    cz, cy, cx = (n // 2 for n in v.shape)
    c = v[: 2 * cz, : 2 * cy, : 2 * cx].reshape(cz, 2, cy, 2, cx, 2)
    d = np.zeros((cz, cy, cx), np.int64)
    s = np.zeros((cz, cy, cx), np.int64)
    for i, j, k in np.ndindex(2, 2, 2):
        corner = c[:, i, :, j, :, k]
        d += corner if (i + j + k) % 2 == 0 else -corner
        s += corner
    ok = s > 0
    return np.abs(d)[ok], s[ok]


def nlf_reference(x, edges=None, min_cells=256):
    """DESIGN §3.12 restated: per bin cells, level_sum, mad, sigma, level; the weighted least-squares (a, b) and the
    number of usable bins.  Same keys as Denoiser.noise_level_function."""
    x = np.asarray(x)
    vols = x[None] if x.ndim == 3 else x
    e = default_edges() if edges is None else np.asarray(edges, np.float64)
    nb = e.size - 1
    ad, s = (np.concatenate(p) for p in zip(*(_cells(v) for v in vols)))
    thr = np.clip(np.ceil(8.0 * e), 0, 524281).astype(np.int64)
    k = np.searchsorted(thr, s, side="right") - 1  # the last k with thr[k] <= s
    cells = np.zeros(nb, np.int64)
    level_sum = np.zeros(nb, np.int64)
    mad = np.full(nb, np.nan)
    for b in range(nb):
        sel = k == b
        cells[b] = int(sel.sum())
        level_sum[b] = int(s[sel].sum())
        if cells[b]:
            mad[b] = np.median(ad[sel])
    sigma = mad / NOISE_C
    level = np.full(nb, np.nan)
    has = cells > 0
    level[has] = level_sum[has] / (8.0 * cells[has])
    W = Sx = Sy = Sxx = Sxy = 0.0
    used = 0
    for b in range(nb):
        if cells[b] < min_cells:
            continue
        w, xx, y = float(cells[b]), float(level[b]), float(sigma[b]) * float(sigma[b])
        W += w
        Sx += w * xx
        Sy += w * y
        Sxx += w * xx * xx
        Sxy += w * xx * y
        used += 1
    a = b_ = float("nan")
    if used >= 2:
        a = (W * Sxy - Sx * Sy) / (W * Sxx - Sx * Sx)
        b_ = (Sy - a * Sx) / W
    return {"cells": cells, "level_sum": level_sum, "level": level, "mad": mad, "sigma": sigma, "a": a, "b": b_,
            "usable": used}


def gat_forward_reference(z, gain, offset, read_sigma):
    q = read_sigma / gain
    qq = q * q
    t = ((np.asarray(z).astype(np.float64) - offset) / gain + 0.375) + qq
    return (2.0 * np.sqrt(np.where(t > 0.0, t, 0.0))).astype(np.float32)


def gat_inverse_reference(D, gain, offset, read_sigma):
    q = read_sigma / gain
    qq = q * q
    d = np.asarray(D, np.float32).astype(np.float64)
    with np.errstate(all="ignore"):
        r = 1.0 / d
        P = 0.25 * d * d + C1 * r - 1.375 * r * r + C2 * r * r * r - 0.125
        lam = P - qq
        lam = np.where(lam > 0.0, lam, 0.0)
        lam = np.where(d <= S15, 0.0, lam)
        return (gain * lam + offset).astype(np.float32)


def pg_volume(shape, seed, gain=2.0, offset=37.0, read_sigma=3.0):
    """(noisy uint16, clean float64): synth.clean_vol as the expected count, z = gain Poisson((c - offset)/gain)
    + N(offset, read_sigma^2), rounded and clipped to uint16."""
    from b4d import synth

    clean = synth.clean_vol(*shape, seed=seed).astype(np.float64)
    rng = np.random.default_rng(seed)
    lam = np.maximum(clean - offset, 0.0) / gain
    z = gain * rng.poisson(lam) + offset + read_sigma * rng.standard_normal(clean.shape)
    return np.clip(np.rint(z), 0, 65535).astype(np.uint16), clean


NLF_KEYS = ("cells", "level_sum", "level", "mad", "sigma")


def _same_nlf(got, ref):
    for key in NLF_KEYS:
        np.testing.assert_array_equal(got[key], ref[key], err_msg=key)
    assert got["usable"] == ref["usable"]
    for key in ("a", "b"):
        assert (np.isnan(got[key]) and np.isnan(ref[key])) or got[key] == ref[key], (key, got[key], ref[key])


@pytest.fixture(scope="module")
def dev():
    import b4d

    return b4d.Denoiser(0)


# ---------------------------------------------------------------- CPU ----
@pytest.mark.parametrize("lam", [0.05, 0.1, 0.2, 0.5, 1.0, 2.0, 5.0])
def test_inverse_is_unbiased_on_poisson_data(lam):
    """The restated inverse of the exact expectation of the forward transform of Poisson(lam) returns lam."""
    from scipy import stats

    k = np.arange(0, 200)
    ef = float(np.sum(stats.poisson.pmf(k, lam) * 2.0 * np.sqrt(k + 0.375)))
    got = float(gat_inverse_reference(np.float32(ef), 1.0, 0.0, 0.0))
    assert abs(got - lam) < 0.01, (lam, got)


def test_inverse_floor_is_continuous():
    below = np.nextafter(np.float32(S15), np.float32(0))
    above = np.nextafter(np.float32(S15), np.float32(10))
    assert gat_inverse_reference(np.array([below, above, -1.0, 0.0]), 1.0, 0.0, 0.0).max() < 1e-6
    # without the floor P would turn positive again below D ~ 0.65
    d = 0.5
    assert 0.25 * d * d + C1 / d - 1.375 / d / d + C2 / d ** 3 - 0.125 > 0


def test_forward_variance_is_stabilised():
    rng = np.random.default_rng(0)
    for lam in (20.0, 200.0, 2000.0):
        z = np.clip(np.rint(2.0 * rng.poisson(lam, 200000) + 37.0 + 3.0 * rng.standard_normal(200000)), 0, 65535)
        f = gat_forward_reference(z.astype(np.uint16), 2.0, 37.0, 3.0)
        assert abs(float(f.std()) - 1.0) < 0.03, (lam, f.std())


def test_restated_nlf_recovers_the_camera():
    """DESIGN §3.12 records these tolerances: on clean_vol(128^3, seed 3) with gain 2, offset 37, read sigma 3 the
    restatement gives a = 2.075, b = -66.66 (true 2, -65) from 13 usable bins."""
    x, _ = pg_volume((128, 128, 128), 3)
    r = nlf_reference(x)
    assert r["usable"] >= 5
    assert abs(r["a"] - 2.0) < 0.25, r["a"]
    assert abs(r["b"] + 65.0) < 15.0, r["b"]


def test_from_nlf():
    import b4d

    m = b4d.PoissonGaussian.from_nlf(2.0, -65.0, 37.0)
    assert m == (2.0, 37.0, 3.0) and m.gain == 2.0 and m.read_sigma == 3.0
    assert b4d.PoissonGaussian.from_nlf(2.0, -100.0, 37.0).read_sigma == 0.0
    np.testing.assert_array_equal(b4d.default_nlf_edges(), default_edges())
    assert b4d.default_nlf_edges().size == 35 and b4d.default_nlf_edges()[-1] == 65536.0


def test_argument_errors_before_touching_the_device():
    import b4d

    x = np.zeros((8, 8, 8), np.uint16)
    good = b4d.PoissonGaussian(2.0, 37.0, 3.0)
    bad_models = [(0.0, 0.0, 1.0), (-1.0, 0.0, 1.0), (np.inf, 0.0, 1.0), (1.0, np.nan, 1.0), (1.0, 0.0, -0.5),
                  (1.0, 0.0, np.inf), (1.0, 2.0), "model"]
    for m in bad_models:
        for call in (lambda: b4d.denoise_vst(x, m), lambda: b4d.gat_forward(x, m),
                     lambda: b4d.gat_inverse(x.astype(np.float32), m)):
            with pytest.raises(ValueError):
                call()
    for sigma in (0.0, -1.0, np.nan, np.inf):
        with pytest.raises(ValueError):
            b4d.denoise_vst(x, good, sigma=sigma)
    for bad in (x.astype(np.float32), x[0], x[None, None]):
        with pytest.raises(ValueError):
            b4d.denoise_vst(bad, good)
    with pytest.raises(ValueError):
        b4d.denoise_vst(x, good, quantize=(0.0, 0.0, 0.5))
    with pytest.raises(ValueError):
        b4d.gat_forward(x.astype(np.float32), good)
    with pytest.raises(ValueError):
        b4d.gat_inverse(x, good)
    for edges in ([0.0], [0.0, 1.0, 1.0], [2.0, 1.0], [0.0, np.inf], [0.0, np.nan, 3.0], np.arange(67.0),
                  [[0.0, 1.0]]):
        with pytest.raises(ValueError):
            b4d.noise_level_function(x, edges=edges)
    for bad in (x.astype(np.int16), x[0]):
        with pytest.raises(ValueError):
            b4d.noise_level_function(bad)
    with pytest.raises(ValueError):
        b4d.noise_level_function(x, min_cells=0)


# ---------------------------------------------------------------- GPU ----
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["pg128", "ragged_odd_w", "batch3", "empty_bins", "one_usable_bin", "fine_edges",
                                  "wide_edges"])
def test_nlf_equals_restatement(dev, case):
    edges, min_cells = None, 256
    if case == "pg128":
        x, _ = pg_volume((128, 128, 128), 3)
    elif case == "ragged_odd_w":  # odd W: the 2-byte load path
        x, _ = pg_volume((37, 50, 61), 5, gain=1.5, offset=100.0, read_sigma=4.0)
    elif case == "batch3":
        x = np.stack([pg_volume((40, 40, 40), s)[0] for s in (6, 7, 8)])
    elif case == "empty_bins":  # bins above the data and a gap: no cells, NaN statistics
        x, _ = pg_volume((48, 48, 48), 9)
        edges, min_cells = [0.0, 30.0, 60.0, 61.0, 400.0, 1e5, 2e5, 3e5], 10
    elif case == "one_usable_bin":
        x, _ = pg_volume((32, 32, 32), 10)
        edges = [0.0, 1e5]
    elif case == "fine_edges":  # fractional and negative edges: ceil(8 e) merges some thresholds
        x = np.random.default_rng(11).integers(0, 9, (20, 22, 24)).astype(np.uint16)
        edges, min_cells = np.linspace(-1.0, 9.0, 65), 1
    else:  # the whole 16-bit range, the top bin holding 65535
        x = np.random.default_rng(12).integers(0, 65536, (24, 26, 28)).astype(np.uint16)
        x[:4, :4, :4] = 65535
        edges, min_cells = np.linspace(0.0, 65536.0, 9), 1
    got = dev.noise_level_function(x, edges=edges, min_cells=min_cells)
    _same_nlf(got, nlf_reference(x, edges, min_cells))
    if case == "empty_bins":
        assert np.all(got["cells"][5:] == 0) and np.all(np.isnan(got["sigma"][5:])) and got["cells"][4] > 0
    if case == "one_usable_bin":
        assert got["usable"] == 1 and np.isnan(got["a"]) and np.isnan(got["b"])


@pytest.mark.gpu
def test_nlf_torch_and_unaligned_input(dev):
    import torch

    x = np.stack([pg_volume((24, 30, 34), s)[0] for s in (13, 14)])
    ref = nlf_reference(x, min_cells=8)
    _same_nlf(dev.noise_level_function(torch.from_numpy(x.view(np.int16)).view(torch.uint16).cuda(), min_cells=8),
              ref)
    flat = torch.zeros(x.size + 1, dtype=torch.int16, device="cuda")
    flat[1:] = torch.from_numpy(x.view(np.int16).reshape(-1)).cuda()
    view = flat[1:].view(torch.uint16).view(x.shape)
    assert view.data_ptr() % 4 == 2  # even W but not 4-byte aligned: the 2-byte load path
    _same_nlf(dev.noise_level_function(view, min_cells=8), ref)


@pytest.mark.gpu
def test_nlf_512_cubed(dev):
    x, _ = pg_volume((512, 512, 512), 4)
    got = dev.noise_level_function(x)
    _same_nlf(got, nlf_reference(x))
    assert got["usable"] >= 5


MODELS = [(2.0, 37.0, 3.0), (1.0, 0.0, 0.0), (0.37, 101.5, 24.0), (5.5, -3.0, 0.25)]


@pytest.mark.gpu
@pytest.mark.parametrize("model", MODELS)
def test_gat_forward_all_uint16_values(dev, model):
    z = np.arange(65536, dtype=np.uint16)
    got = dev.gat_forward(z, model)
    assert got.dtype == np.float32
    np.testing.assert_array_equal(got, gat_forward_reference(z, *model))


@pytest.mark.gpu
@pytest.mark.parametrize("model", MODELS)
def test_gat_inverse_bit_exact(dev, model):
    s = np.float32(S15)
    near = [s]
    for _ in range(4):
        near += [np.nextafter(near[-1], np.float32(10)), np.nextafter(near[0 if len(near) < 2 else -2], np.float32(0))]
    D = np.concatenate([np.array(near + [0.0, -0.0, -1.0, -1e30, 0.5, 0.65, 1.0, 1e-30, 1e20, 3e38], np.float32),
                        np.random.default_rng(1).uniform(-2.0, 600.0, 100003).astype(np.float32),
                        gat_forward_reference(np.arange(65536, dtype=np.uint16), *model)])
    got = dev.gat_inverse(D, model)
    np.testing.assert_array_equal(got, gat_inverse_reference(D, *model))


@pytest.mark.gpu
def test_gat_unaligned_device_pointers(dev):
    import torch

    model = MODELS[0]
    z = np.random.default_rng(2).integers(0, 65536, 10001).astype(np.uint16)
    buf = torch.zeros(z.size + 1, dtype=torch.int16, device="cuda")
    buf[1:] = torch.from_numpy(z.view(np.int16)).cuda()
    zv = buf[1:].view(torch.uint16)
    assert zv.data_ptr() % 4 == 2
    f = dev.gat_forward(zv, model)
    np.testing.assert_array_equal(f.cpu().numpy(), gat_forward_reference(z, *model))
    fb = torch.zeros(z.size + 1, dtype=torch.float32, device="cuda")
    fb[1:] = f
    fv = fb[1:]
    assert fv.data_ptr() % 16 == 4
    np.testing.assert_array_equal(dev.gat_inverse(fv, model).cpu().numpy(),
                                  gat_inverse_reference(f.cpu().numpy(), *model))


@pytest.mark.gpu
def test_denoise_vst_equals_the_composition(dev):
    import b4d

    x, _ = pg_volume((40, 44, 48), 14)
    m = b4d.PoissonGaussian(2.0, 37.0, 3.0)
    comp = dev.gat_inverse(dev.denoise(dev.gat_forward(x, m), 1.0), m)
    got = dev.denoise_vst(x, m)
    assert got.dtype == np.float32 and got.shape == x.shape
    np.testing.assert_array_equal(got, comp)
    # another post-transform sigma
    np.testing.assert_array_equal(dev.denoise_vst(x, m, sigma=1.3),
                                  dev.gat_inverse(dev.denoise(dev.gat_forward(x, m), 1.3), m))


@pytest.mark.gpu
def test_denoise_vst_equals_the_oracle_mirror(dev, oracle_lib):
    x, _ = pg_volume((24, 26, 28), 15)
    m = (2.0, 37.0, 3.0)
    mirror = oracle_lib.Oracle("mirror").denoise(gat_forward_reference(x, *m), 1.0)
    np.testing.assert_array_equal(dev.denoise_vst(x, m), gat_inverse_reference(mirror, *m))


@pytest.mark.gpu
def test_denoise_vst_batch_equals_patches_and_torch(dev):
    import torch

    m = (1.5, 90.0, 5.0)
    x = np.stack([pg_volume((30, 32, 34), s, gain=1.5, offset=90.0, read_sigma=5.0)[0] for s in (16, 17, 18)])
    got = dev.denoise_vst(x, m)
    for i in range(3):
        np.testing.assert_array_equal(got[i], dev.denoise_vst(x[i], m))
    xt = torch.from_numpy(x.view(np.int16)).view(torch.uint16).cuda()
    gt = dev.denoise_vst(xt, m)
    assert gt.is_cuda and gt.dtype == torch.float32
    np.testing.assert_array_equal(gt.cpu().numpy(), got)


@pytest.mark.gpu
@pytest.mark.parametrize("truncate", [False, True])
def test_denoise_vst_q16_equals_quantize(dev, truncate):
    import torch

    x, _ = pg_volume((36, 40, 44), 19)
    m = (2.0, 37.0, 3.0)
    y = dev.denoise_vst(x, m)
    for q in ((37.0, 0.0, 1.0), (37.0, 5.0, 3.5)):
        want = dev.quantize(y, *q, truncate=truncate)
        got = dev.denoise_vst(x, m, quantize=q + (truncate,))
        assert got.dtype == np.uint16
        np.testing.assert_array_equal(got, want)
        gt = dev.denoise_vst(torch.from_numpy(x.view(np.int16)).view(torch.uint16).cuda(), m, quantize=q + (truncate,))
        np.testing.assert_array_equal(gt.cpu().numpy(), want)


@pytest.mark.gpu
def test_vst_beats_one_background_sigma(dev):
    """On shot-noise-dominated counts, denoising through the GAT with the model estimated from the data has a lower
    RMSE against the clean signal than denoising at the one sigma of noise_sigma (DESIGN §8 records both)."""
    import b4d

    x, clean = pg_volume((128, 128, 128), 3)
    nlf = dev.noise_level_function(x)
    model = b4d.PoissonGaussian.from_nlf(nlf["a"], nlf["b"], dev.tile_stats(x)["offset"])
    vst = dev.denoise_vst(x, model)
    base = dev.denoise(x, float(dev.noise_sigma(x)["sigma"]))
    rmse_vst = float(np.sqrt(np.mean((vst - clean) ** 2)))
    rmse_base = float(np.sqrt(np.mean((base - clean) ** 2)))
    assert rmse_vst < rmse_base, (rmse_vst, rmse_base)
