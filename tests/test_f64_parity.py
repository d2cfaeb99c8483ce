"""The float32 path against the plain float64 oracle (DESIGN §5) beyond the default case: every matching-map regime
of DESIGN §3.1, every filter instantiation, stage 1 alone as well as both stages, the Poisson-Gaussian (VST) path at
its operating point, and power-of-two scale equivariance.

The float32 mirror (Oracle("mirror")) follows the kernels operation for operation, so a mistake the two share passes
every bit-exact test.  The float64 oracle (Oracle("f64"): dense orthonormal transforms, float64 weights and sums)
shares no arithmetic with them.  Bars, relative to sigma so that they carry over to float data at any scale (at
sigma = 24 they are 0.5 and 0.05 counts):

* rel-L2 <= 1e-3;
* both stages: max-abs <= 0.5 sigma / 24 except under a stage-2 group whose match list differs between the float32 and
  the float64 pipeline (oracle/parity_util.flipped_support), and <= 0.05 sigma / 24 away from every such group;
* stage 1 alone: max-abs <= 0.01 sigma.  Stage 1 has no stage-2 groups to flip, but a hard-threshold decision can flip
  where a coefficient lies within float32 rounding of lambda sigma.  The test does not localise such flips: its volumes
  and seeds are chosen so that none occurs.  Measured on the map regimes: at most 1e-3 sigma, a few float32 spacings of
  the output where the range is 4000 sigma or the level 4000 sigma and more, and 5e-6 sigma elsewhere.

CPU tests hold the float32 mirror to these bars.  GPU tests hold the device to the mirror bit for bit and to the bars.

uint16 input is its own matching image and aggregates at unit scale whatever sigma is; the map rule does not apply to
it.  At sigma < 1 this costs accuracy against the float64 oracle: on synth.vol(20, 21, 22, seed 7) at sigma = 0.5,
both stages, the mirror is up to 3e-4 (6e-4 sigma) from it.
"""
import functools

import numpy as np
import pytest

from b4d import synth

SHAPE = (20, 21, 22)
REL_L2 = 1e-3
STAGE1_MAX_ABS = 0.01  # in units of sigma


def rel_l2(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b.astype(np.float64)) / max(np.linalg.norm(b), 1e-30))


@functools.lru_cache(maxsize=None)
def _structure():
    """A part of the clean synthetic field with fibres and a blob, on SHAPE, scaled to [0, 1]."""
    c = synth.clean_vol(*SHAPE, 3, z0=36, y0=96, x0=24).astype(np.float64)
    return (c - c.min()) / (c.max() - c.min())


def _noise(seed):
    return np.random.default_rng(seed).standard_normal(SHAPE)


def _sigma_at(e):
    """The sigma whose sigma-bound scale floor(log2(64 / sigma)) is 2^e, 0.415 away from the floor's steps."""
    return 0.75 * 2.0 ** (6 - e)


def _float_case(sigma, amplitude, seed, dc=0.0):
    """amplitude * structure + N(dc, sigma), float32: non-integral data."""
    return (dc + amplitude * _structure() + sigma * _noise(seed)).astype(np.float32), sigma


def _counts(seed=7):
    return synth.vol(*SHAPE, seed=seed)


# name -> (data, sigma) and the map DESIGN §3.1 gives it: (integral, log2 scale, centred)
REGIMES = {
    "u16_counts": (lambda: (_counts(), 24.0), (True, 0, False)),
    "counts_minus_offset": (lambda: (_counts().astype(np.float32) - np.float32(36.37), 24.0), (True, 0, False)),
    **{"sigma_scale_%d" % e: (lambda e=e: _float_case(_sigma_at(e), 8 * _sigma_at(e), 10 + e), (False, e, False))
       for e in (-5, 0, 6, 12, 18)},
    # sigma at 2^6 steps would need more than 16 bits for this range: the range sets the scale
    "range_bound": (lambda: _float_case(0.75, 3000.0, 31), (False, 4, False)),
    "dc_counts": (lambda: (_counts().astype(np.float32) + np.float32(2.0e5), 24.0), (True, 0, True)),
    "dc_float": (lambda: _float_case(0.05, 0.4, 32, dc=200.0), (False, 10, True)),
    # the whole range, noise included, within 1/64 of one integer
    "noise_3e-3": (lambda: _float_case(3e-3, 0.0, 41), (False, 14, False)),
    "noise_1e-3": (lambda: _float_case(1e-3, 0.0, 42), (False, 15, False)),
    "noise_1e-4": (lambda: _float_case(1e-4, 0.0, 43), (False, 19, False)),
    "noise_1e-5": (lambda: _float_case(1e-5, 0.0, 44), (False, 22, False)),
    "dim_structure": (lambda: _float_case(2e-3, 4e-3, 45), (False, 14, False)),
    "tiny_structure": (lambda: _float_case(1e-5, 1e-4, 46), (False, 22, False)),
}


def _map(oracle_lib, z, sigma):
    integral, scale, centre = oracle_lib.match_map(z, sigma)
    e = int(np.log2(scale))
    assert scale == 2.0 ** e
    return integral, e, centre != 0.0


def assert_f64_bar(y, f, sigma, stages, om=None, of=None, Ns=11):
    """y (float32 path) against f (float64 oracle) within the bars of the module docstring.  Two stages need the
    float32 and the float64 oracle handles of the call, om and of, for their stage-2 match lists."""
    from oracle import parity_util

    assert rel_l2(y, f) <= REL_L2
    if stages == 1:
        err = float(np.abs(y.astype(np.float64) - f).max())
        assert err <= STAGE1_MAX_ABS * sigma, "stage 1: max-abs %g = %g sigma" % (err, err / sigma)
        return
    parity_util.check_against_f64(y, f, om.stage2_matches(y.shape), of.stage2_matches(y.shape),
                                  max_abs=0.5 * sigma / 24.0, quiet_abs=0.05 * sigma / 24.0, Ns=Ns)


# ---------------------------------------------------------------------------------------------------------- CPU --
@pytest.mark.parametrize("stages", [1, 2])
@pytest.mark.parametrize("name", list(REGIMES))
def test_mirror_meets_the_f64_bar_in_every_map_regime(name, stages, oracle_lib):
    make, want = REGIMES[name]
    z, sigma = make()
    assert _map(oracle_lib, z, sigma) == want
    om, of = oracle_lib.Oracle("mirror", stages=stages), oracle_lib.Oracle("f64", stages=stages)
    assert_f64_bar(om.denoise(z, sigma), of.denoise(z, sigma), sigma, stages, om, of)


# sigma 0.75 * 2^m: away from the steps of floor(log2(64 / sigma)) at every 2^k
EQUIVARIANCE = {
    "non_integral": lambda: _float_case(0.75, 6.0, 51, dc=0.3),
    "small_range": lambda: _float_case(0.75 * 2.0 ** -10, 1.5 * 2.0 ** -10, 52),
}


@functools.lru_cache(maxsize=None)
def _mirror_at_unit_scale(data):
    from oracle import np_oracle

    z, sigma = EQUIVARIANCE[data]()
    return z, sigma, np_oracle.Oracle("mirror").denoise(z, sigma)


@pytest.mark.parametrize("k", [-12, -6, -1, 1, 6, 12])
@pytest.mark.parametrize("data", list(EQUIVARIANCE))
def test_mirror_is_power_of_two_scale_equivariant(data, k, oracle_lib):
    """mirror(2^k z, 2^k sigma) == 2^k mirror(z, sigma), bit for bit: with the map's scale shifted by 2^-k, the
    matching image, the fixed-point terms and every float32 operation scale exactly."""
    z, sigma, y = _mirror_at_unit_scale(data)
    s = np.float32(2.0 ** k)
    zs, sigma_s = z * s, sigma * 2.0 ** k
    integral, e, centred = _map(oracle_lib, z, sigma)
    assert not integral and not centred
    assert _map(oracle_lib, zs, sigma_s) == (False, e - k, False)
    ys = oracle_lib.Oracle("mirror").denoise(zs, sigma_s)
    assert np.array_equal(ys, y * s), "max-abs %g sigma" % (np.abs(ys / s - y).max() / sigma)


# ---------------------------------------------------------------------------------------------------------- GPU --
@pytest.fixture(scope="module")
def b4d_mod():
    import b4d

    return b4d


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(REGIMES))
def test_device_meets_the_f64_bar_in_every_map_regime(name, b4d_mod, oracle_lib):
    z, sigma = REGIMES[name][0]()
    d = b4d_mod.Denoiser(0)
    try:
        for stages in (1, 2):
            d.set_profile(None, stages)
            y = d.denoise(z, sigma)
            om, of = oracle_lib.Oracle("mirror", stages=stages), oracle_lib.Oracle("f64", stages=stages)
            m = om.denoise(z, sigma)
            assert np.array_equal(y, m), "stages %d: max-abs %g vs the mirror" % (stages, np.abs(y - m).max())
            assert_f64_bar(y, of.denoise(z, sigma), sigma, stages, om, of)
    finally:
        d.close()


def _window(ns):
    return (ns // 2,) * 3


# (Denoiser profile, oracle profile): the cases of test_gpu_parity.py::test_other_profiles_bit_exact_vs_mirror, then
# group sizes 1, 2 and 4 in both stages at windows 3 and 5
PROFILES = [
    (dict(search_window_ht=(7, 7, 7), search_window_wiener=(7, 7, 7)), dict(search_ht=15, search_wie=15)),
    (dict(search_window_ht=(6, 6, 6), search_window_wiener=(3, 3, 3)), dict(search_ht=13, search_wie=7)),
    (dict(max_stack_size_ht=32, max_stack_size_wiener=16), dict(k_ht=32, k_wie=16)),
    (dict(max_stack_size_ht=8, max_stack_size_wiener=8), dict(k_ht=8, k_wie=8)),
    (dict(max_stack_size_ht=1, max_stack_size_wiener=2, search_window_ht=(1, 1, 1)), dict(k_ht=1, k_wie=2, search_ht=3)),
    (dict(beta=0.0, lambda_thr=3.1, tau_match_ht=1.5), dict(kaiser_beta=0.0, lambda_ht=3.1, tau_ht=1.5)),
] + [
    (dict(max_stack_size_ht=kh, max_stack_size_wiener=kw, search_window_ht=_window(ns), search_window_wiener=_window(ns)),
     dict(k_ht=kh, k_wie=kw, search_ht=ns, search_wie=ns))
    for kh, kw, ns in ((1, 2, 3), (2, 4, 3), (4, 1, 3), (1, 4, 5), (2, 1, 5), (4, 2, 5))
]


@pytest.mark.gpu
@pytest.mark.parametrize("kw,okw", PROFILES)
def test_other_profiles_meet_the_f64_bar(kw, okw, b4d_mod, oracle_lib):
    rng = np.random.default_rng(5)
    vols = [synth.vol(22, 25, 28, seed=21), np.clip(rng.normal(300, 24, (17, 18, 20)), 0, 65535).astype(np.uint16)]
    d = b4d_mod.Denoiser(0, b4d_mod.BM4DProfile(**kw))
    try:
        for vol in vols:
            for stages in (1, 2):
                d.set_profile(b4d_mod.BM4DProfile(**kw), stages)
                y = d.denoise(vol, 24.0)
                om = oracle_lib.Oracle("mirror", stages=stages, **okw)
                of = oracle_lib.Oracle("f64", stages=stages, **okw)
                assert np.array_equal(y, om.denoise(vol, 24.0)), "stages %d" % stages
                assert_f64_bar(y, of.denoise(vol, 24.0), 24.0, stages, om, of, Ns=okw.get("search_wie", 11))
    finally:
        d.close()


@pytest.mark.gpu
def test_coloured_noise_with_other_group_sizes_meets_the_f64_bar(b4d_mod, oracle_lib):
    """Coloured noise with 8-block hard-threshold and 16-block Wiener groups, float32 and uint16 input."""
    from test_oracle_bm4d import _coloured_case

    psd, _, z = _coloured_case((24, 28, 32))
    s, a, b = b4d_mod.noise_model_from_psd(psd)
    zu = np.clip(np.rint(z + 200.0), 0, 65535).astype(np.uint16)
    d = b4d_mod.Denoiser(0, b4d_mod.BM4DProfile(max_stack_size_ht=8, max_stack_size_wiener=16))
    d.set_noise_model(a, b)
    try:
        for x in (z, zu):
            om, of = oracle_lib.Oracle("mirror", k_ht=8, k_wie=16), oracle_lib.Oracle("f64", k_ht=8, k_wie=16)
            om.set_noise_model(a, b)
            of.set_noise_model(a, b)
            y = d.denoise(x, s)
            assert np.array_equal(y, om.denoise(x, s))
            assert_f64_bar(y, of.denoise(x, s), s, 2, om, of)
    finally:
        d.close()


@pytest.mark.gpu
def test_denoise_vst_meets_the_f64_bar_before_the_inverse(b4d_mod, oracle_lib):
    """denoise_vst on a 128^3 Poisson-Gaussian volume (gain 2, offset 37, read sigma 3) is the restated inverse of
    the device's float32 denoise of the forward transform at sigma 1, and that pre-inverse volume is within the bar
    of the float64 oracle on the same forward transform."""
    from test_poisson_gaussian import gat_forward_reference, gat_inverse_reference, pg_volume

    x, _ = pg_volume((128, 128, 128), 3)
    m = (2.0, 37.0, 3.0)
    d = b4d_mod.Denoiser(0)
    try:
        fwd = d.gat_forward(x, m)
        np.testing.assert_array_equal(fwd, gat_forward_reference(x, *m))
        pre = d.denoise(fwd, 1.0)
        np.testing.assert_array_equal(d.denoise_vst(x, m), gat_inverse_reference(pre, *m))
    finally:
        d.close()
    assert _map(oracle_lib, fwd, 1.0) == (False, 6, False)
    om, of = oracle_lib.Oracle("mirror"), oracle_lib.Oracle("f64")
    assert np.array_equal(pre, om.denoise(fwd, 1.0))
    assert_f64_bar(pre, of.denoise(fwd, 1.0), 1.0, 2, om, of)


@pytest.mark.gpu
@pytest.mark.parametrize("side", [256, 1024])
def test_device_is_power_of_two_scale_equivariant(side, b4d_mod, oracle_lib):
    """denoise(2^k z, 2^k sigma) == 2^k denoise(z, sigma) on the device, bit for bit, k = -8 and 8, on counts made
    non-integral (sigma 0.024, scale 2^11) and on the same counts squeezed into a range below 1/64 (sigma 1.2e-5,
    scale 2^22).  256^3: synth.vol; 1024^3: the benchmark volume."""
    import torch

    import bench

    dev = torch.device("cuda", 0)
    if side == 256:
        counts = torch.from_numpy(synth.vol(side, side, side, seed=3)).to(dev)
    else:
        counts = bench.make_slab_device(side, 0, side, dev)
    d = b4d_mod.Denoiser(0)
    try:
        for factor, sigma, e in ((1e-3, 24e-3, 11), (5e-7, 24 * 5e-7, 22)):
            z = (counts.float() - 37.0) * factor
            # the map depends on the first value and on extremes: a corner that holds both gives the volume's map
            probe = z[:8, :8, :8].cpu().numpy()
            probe.flat[1:3] = [float(z.min()), float(z.max())]
            assert _map(oracle_lib, probe, sigma) == (False, e, False)
            y = d.denoise(z, sigma)
            for k in (-8, 8):
                s = 2.0 ** k
                assert torch.equal(d.denoise(z * s, sigma * s), y * s), (factor, k)
            del z, y
    finally:
        d.close()
        del counts
        torch.cuda.empty_cache()
