"""z-slab forms of the Poisson-Gaussian (VST) path (DESIGN §3.12, map rule): a slab given the value set and the first
voxel of the whole volume equals the whole volume's denoise_vst bit for bit, in the no-exchange, exchange and oversize
forms.  Ranks are emulated by one handle each on one GPU.  CPU tests: the header against the binding's table, the new
Denoiser methods against a fake library, and the sharded orchestration against a fake denoiser."""
import ctypes
import math

import numpy as np
import pytest

from test_binding import FakeLib, _prototypes
from test_poisson_gaussian import gat_forward_reference, pg_volume


# ------------------------------------------------------------------ NumPy restatement of the map rule ----
def match_scale(values, first, model, sigma):
    """(scale, centred) that derive_match_map and the centring of prepare_f32 give on the GAT-forwarded list
    [f(first), f(u) for u in values] (csrc/b4d_api.cu; oracle derive_match_map)."""
    z = gat_forward_reference(np.concatenate([[first], np.asarray(values, np.uint16)]).astype(np.uint16), *model)
    z = z.astype(np.float64)
    c = np.rint(z[0]) - z[0]
    v = z + c
    dev = np.max(np.abs(v - np.rint(v)))
    lo, hi, zlo, zhi = np.rint(v).min(), np.rint(v).max(), z.min(), z.max()
    if dev <= min(1.0, float(np.float32(sigma))) / 64.0 and hi - lo <= 65535.0:
        scale = 1.0
    else:
        e_range = math.floor(math.log2(65535.0 / max(zhi - zlo, 1e-30)))
        e_sigma = math.floor(math.log2(64.0 / float(np.float32(sigma))))
        scale = 2.0 ** min(e_range, e_sigma)
    return scale, max(abs(zlo), abs(zhi)) * scale > 131072.0


def value_hist(x):
    return np.bincount(np.asarray(x).ravel(), minlength=65536).astype(np.int64)


def teeth_volume():
    """Counts at a small gain with one bright structure in the lower planes: the whole volume's matching scale is
    range-limited, the upper planes alone are sigma-limited."""
    x, _ = pg_volume((90, 24, 28), 41, gain=0.1, offset=37.0, read_sigma=3.0)
    rng = np.random.default_rng(41)
    x[0:4, 4:14, 5:15] = np.clip(40000 + rng.normal(0, 70, (4, 10, 10)), 0, 65535).astype(np.uint16)
    return x, (0.1, 37.0, 3.0)


def slabs_no_exchange(dn, x, model, world, sigma=1.0, quantize=None, vst_hist=None, first=None):
    from b4d.sharding import halo_planes, slab_plan

    D = x.shape[0]
    vh = value_hist(x) if vst_hist is None else vst_hist
    first = int(x[0, 0, 0]) if first is None else first
    parts = []
    for r in range(world):
        ob, oe, zb, ze = slab_plan(D, world, r, halo_planes())
        parts.append(dn.denoise_slab_vst(x[zb:ze], zb, D, ob, oe, model, vh, first, sigma, quantize=quantize))
    return np.concatenate(parts, 0)


@pytest.fixture(scope="module")
def dn():
    import b4d

    d = b4d.Denoiser(0)
    yield d
    d.close()


# ---------------------------------------------------------------------------------------------------------- GPU --
@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_no_exchange_slabs_equal_the_whole_volume(dn, world):
    x, m = teeth_volume()
    whole = dn.denoise_vst(x, m)
    np.testing.assert_array_equal(slabs_no_exchange(dn, x, m, world), whole)
    for q in ((37.0, 0.0, 1.0, False), (37.0, 5.0, 3.5, True)):
        np.testing.assert_array_equal(slabs_no_exchange(dn, x, m, world, quantize=q), dn.denoise_vst(x, m, quantize=q))


@pytest.mark.gpu
def test_a_slab_with_its_own_value_set_differs():
    """The precondition that gives the slab tests their teeth: the upper planes alone have another matching scale,
    and a slab denoised with its own value set (or as a volume of its own) differs from the whole volume there."""
    import b4d
    from b4d.sharding import halo_planes, slab_plan

    x, m = teeth_volume()
    ob, oe, zb, ze = slab_plan(90, 2, 1, halo_planes())
    top = x[zb:ze]
    whole_scale, _ = match_scale(np.unique(x), x[0, 0, 0], m, 1.0)
    slab_scale, _ = match_scale(np.unique(top), top[0, 0, 0], m, 1.0)
    assert whole_scale == 32.0 and slab_scale == 64.0, (whole_scale, slab_scale)
    dn = b4d.Denoiser(0)
    try:
        whole = dn.denoise_vst(x, m)[ob:oe]
        own_set = dn.denoise_slab_vst(top, zb, 90, ob, oe, m, value_hist(top), int(top[0, 0, 0]))
        assert not np.array_equal(own_set, whole)
        assert not np.array_equal(dn.denoise_vst(top, m)[ob - zb :], whole)
        np.testing.assert_array_equal(dn.denoise_slab_vst(top, zb, 90, ob, oe, m, value_hist(x), int(x[0, 0, 0])),
                                      whole)
    finally:
        dn.close()


def _exchange_ranks(x, m, world):
    import b4d
    from b4d.sharding import exchange_halo, slab_plan

    D, h = x.shape[0], exchange_halo(11, 11)
    vh, first = value_hist(x), int(x[0, 0, 0])
    ranks = []
    for r in range(world):
        ob, oe, zb, ze = slab_plan(D, world, r, h)
        d = b4d.Denoiser(0)
        d.slab_stage1_vst(x[zb:ze], zb, D, m, vh, first)
        ranks.append((d, ob, oe, zb, ze))
    return ranks, h


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_exchange_staging_copies_equal_the_whole_volume(dn, world):
    x, m = teeth_volume()
    whole = dn.denoise_vst(x, m)
    wq = dn.denoise_vst(x, m, quantize=(37.0, 0.0, 2.0))
    for q in (None, (37.0, 0.0, 2.0)):
        ranks, h = _exchange_ranks(x, m, world)
        sends = [(d.slab_basic(ob - zb, h), d.slab_basic(oe - zb - h, h)) for d, ob, oe, zb, ze in ranks]
        parts = []
        for r, (d, ob, oe, zb, ze) in enumerate(ranks):
            if r > 0:
                d.slab_set_basic(0, sends[r - 1][1])
            if r < world - 1:
                d.slab_set_basic(oe - zb, sends[r + 1][0])
            parts.append(d.slab_stage2(ob, oe, quantize=q))
            d.close()
        np.testing.assert_array_equal(np.concatenate(parts, 0), whole if q is None else wq)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_exchange_in_place_overlapped_equals_the_whole_volume(dn, world):
    """The device path of sharding.denoise_slab_exchange: part 1 of the stage-2 front end is launched before the
    neighbours' planes are written into the basic estimate in place."""
    import torch

    x, m = teeth_volume()
    whole = dn.denoise_vst(x, m)
    ranks, h = _exchange_ranks(x, m, world)
    dev = torch.device("cuda", 0)
    views = [d.slab_basic_tensor(dev) for d, *_ in ranks]
    for d, ob, oe, zb, ze in ranks:
        d.slab_stage2_begin(ob, oe)
    sends = [(v[ob - zb : ob - zb + h].clone(), v[oe - zb - h : oe - zb].clone())
             for v, (d, ob, oe, zb, ze) in zip(views, ranks)]
    for r, (v, (d, ob, oe, zb, ze)) in enumerate(zip(views, ranks)):
        if r > 0:
            v[0:h].copy_(sends[r - 1][1])
        if r < world - 1:
            v[oe - zb : oe - zb + h].copy_(sends[r + 1][0])
    torch.cuda.synchronize()
    parts = [d.slab_stage2(ob, oe, device=dev).cpu().numpy() for d, ob, oe, zb, ze in ranks]
    for d, *_ in ranks:
        d.close()
    np.testing.assert_array_equal(np.concatenate(parts, 0), whole)


def _tall():
    x, _ = pg_volume((100, 24, 28), 43, gain=2.0, offset=37.0, read_sigma=3.0)
    return x, (2.0, 37.0, 3.0)


@pytest.mark.gpu
def test_oversize_volumes_equal_one_pass():
    import torch

    import b4d

    x, m = _tall()
    one, big = b4d.Denoiser(0), b4d.Denoiser(0)
    try:
        big.set_pass_voxels(60 * 24 * 28)  # 13 slabs of 8 owned planes
        xt = torch.from_numpy(x.view(np.int16)).view(torch.uint16).cuda()
        for q in (None, (37.0, 0.0, 1.0, False), (37.0, 5.0, 3.5, True)):
            want = one.denoise_vst(x, m, quantize=q)
            launches_one = sum(n for _, n in one.last_timings().values())
            np.testing.assert_array_equal(big.denoise_vst(x, m, quantize=q), want)
            assert sum(n for _, n in big.last_timings().values()) > 5 * launches_one
            np.testing.assert_array_equal(big.denoise_vst(xt, m, quantize=q).cpu().numpy(), want)
        x2 = np.stack([x, pg_volume((100, 24, 28), 44)[0]])
        np.testing.assert_array_equal(big.denoise_vst(x2, m), one.denoise_vst(x2, m))
        big.set_pass_voxels(40 * 24 * 28)  # two halos of 26 planes do not fit
        with pytest.raises(ValueError):
            big.denoise_vst(x, m)
    finally:
        one.close()
        big.close()


def _corner_cases():
    rng = np.random.default_rng(45)
    const = np.full((64, 20, 24), 500, np.uint16)
    two = rng.choice(np.array([100, 3000], np.uint16), (64, 20, 24))
    dc, _ = pg_volume((64, 20, 24), 46)
    return [("constant", const, (2.0, 37.0, 3.0), 1.0), ("two_valued", two, (2.0, 37.0, 3.0), 1.0),
            ("centred", dc, (1.0, -4.0e6, 3.0), 1.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c[0] for c in _corner_cases()])
def test_map_corner_cases_slabbed_equal_whole(dn, case):
    name, x, m, sigma = [c for c in _corner_cases() if c[0] == case][0]
    scale, centred = match_scale(np.unique(x), x[0, 0, 0], m, sigma)
    assert (scale == 1.0) == (name == "constant") and centred == (name == "centred"), (scale, centred)
    whole = dn.denoise_vst(x, m, sigma)
    for world in (2, 3):
        np.testing.assert_array_equal(slabs_no_exchange(dn, x, m, world, sigma), whole)


@pytest.mark.gpu
def test_pipelined_host_output_equals_device_output():
    """A deep volume whose result goes to host memory is normalised, inverted and copied out chunk by chunk while the
    filter still runs; pageable and pinned outputs equal the device output."""
    import torch

    import b4d

    x, _ = pg_volume((208, 16, 20), 47)
    m = (2.0, 37.0, 3.0)
    d = b4d.Denoiser(0)
    try:
        d.set_pipeline_min_voxels(0)
        xt = torch.from_numpy(x.view(np.int16)).view(torch.uint16).cuda()
        for q in (None, (37.0, 0.0, 2.0)):
            dev_out = d.denoise_vst(xt, m, quantize=q).cpu().numpy()
            np.testing.assert_array_equal(d.denoise_vst(x, m, quantize=q), dev_out)
            assert d.last_timings()["norm2"][1] > 1  # the chunked normalise ran
            vh, first = value_hist(x), int(x[0, 0, 0])
            pinned = torch.empty(x.shape, dtype=torch.float32 if q is None else torch.int16, pin_memory=True).numpy()
            pinned = pinned if q is None else pinned.view(np.uint16)
            got = d.denoise_slab_vst(x, 0, 208, 0, 208, m, vh, first, out=pinned, quantize=q)
            assert got is pinned
            np.testing.assert_array_equal(pinned, dev_out)
            np.testing.assert_array_equal(d.denoise_slab_vst(x, 0, 208, 0, 208, m, vh, first, quantize=q), dev_out)
    finally:
        d.close()


@pytest.mark.gpu
def test_rejections(dn):
    x, m = teeth_volume()
    vh, first = value_hist(x), int(x[0, 0, 0])
    slab = x[:40]
    absent_first = vh.copy()
    absent_first[first] = 0
    with pytest.raises(ValueError, match="first_value"):
        dn.denoise_slab_vst(slab, 0, 90, 0, 30, m, absent_first, first)
    missing = vh.copy()
    missing[int(slab[2, 8, 8])] = 0  # a value of the bright block
    with pytest.raises(ValueError, match="value_hist"):
        dn.denoise_slab_vst(slab, 0, 90, 0, 30, m, missing, first)
    with pytest.raises(ValueError, match="value_hist"):
        dn.slab_stage1_vst(slab, 0, 90, m, missing, first)
    with pytest.raises(ValueError, match="65536"):
        dn.denoise_slab_vst(slab, 0, 90, 0, 30, m, vh[:-1], first)
    negative = vh.copy()
    negative[7] = -1
    with pytest.raises(ValueError, match="negative"):
        dn.denoise_slab_vst(slab, 0, 90, 0, 30, m, negative, first)
    # the handle is still usable
    np.testing.assert_array_equal(slabs_no_exchange(dn, x, m, 2), dn.denoise_vst(x, m))


def _timing_case(name):
    import b4d

    d = b4d.Denoiser(0)
    x, m = _tall()
    vh, first = value_hist(x), int(x[0, 0, 0])
    if name == "vst_slab":
        return d, lambda: d.denoise_slab_vst(x[20:80], 20, 100, 40, 60, m, vh, first)
    if name == "vst_slab_q16":
        return d, lambda: d.denoise_slab_vst(x[20:80], 20, 100, 40, 60, m, vh, first, quantize=(37.0, 0.0, 2.0))
    if name == "vst_two_call_begin":
        def call():
            d.slab_stage1_vst(x[20:80], 20, 100, m, vh, first)
            d.slab_stage2_begin(40, 60)
            d.slab_stage2(40, 60)
        return d, call
    if name == "vst_oversize":
        d.set_pass_voxels(60 * 24 * 28)
        return d, lambda: d.denoise_vst(x, m)
    raise KeyError(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["vst_slab", "vst_slab_q16", "vst_two_call_begin", "vst_oversize"])
def test_booked_launches_equal_the_profiler(name, tmp_path):
    from test_timings import _launches, _profiled_kernels

    d, call = _timing_case(name)
    try:
        kernels = _profiled_kernels(call, tmp_path)
        assert _launches(d) == kernels, (kernels, d.last_timings())
    finally:
        d.close()


# ---------------------------------------------------------------------------------------------------------- CPU --
VST_PROTOS = _prototypes("b4d_vst_slab.h")
VST_PARAMS = {name: [n for _, n in params] for name, (_, params) in VST_PROTOS.items()}


def test_header_matches_the_table():
    from b4d import _lib

    scalars = {"int64_t": ctypes.c_int64, "int": ctypes.c_int, "float": ctypes.c_float, "double": ctypes.c_double}
    assert sorted(_lib.VST_SLAB_EXPORTS) == sorted(VST_PROTOS) and len(VST_PROTOS) == 3
    for name, (ret, params) in VST_PROTOS.items():
        restype, argtypes = _lib.VST_SLAB_SIGNATURES[name]
        assert ret == "int" and restype is ctypes.c_int
        assert argtypes == [ctypes.c_void_p if t == "*" else scalars[t] for t, _ in params], name
    assert not set(_lib.VST_SLAB_SIGNATURES) & set(_lib.SIGNATURES)


def _fake_denoiser():
    import os

    import b4d
    from b4d import _lib

    fake = FakeLib()
    fake.hists = []  # the value set each call was given, read while the call runs

    def snapshot(name, fn):
        def call(*args):
            at = args[VST_PARAMS[name].index("value_hist")]
            fake.hists.append(np.ctypeslib.as_array((ctypes.c_int64 * 65536).from_address(at)).copy())
            return fn(*args)
        return call

    for name, (_, argtypes) in _lib.VST_SLAB_SIGNATURES.items():
        setattr(fake, name, snapshot(name, fake._fn(name, argtypes, 0)))
    d = object.__new__(b4d.Denoiser)
    d.lib, d.device, d.profile, d._stages = fake, 0, b4d.BM4DProfile(), 2
    d._h, d._pid = ctypes.c_void_p(0x1000), os.getpid()
    return d, fake


def _args(fake, name):
    called, args = fake.calls[-1]
    assert called == name
    return dict(zip(VST_PARAMS[name], args))


def test_denoiser_methods_on_a_fake_library():
    import torch

    import b4d

    d, fake = _fake_denoiser()
    slab = np.arange(9 * 7 * 8, dtype=np.uint16).reshape(9, 7, 8)
    vh = value_hist(slab)
    model = b4d.PoissonGaussian(2.0, 37.0, 3.0)
    for x in (slab, torch.from_numpy(slab.view(np.int16)).view(torch.uint16)):
        out = d.denoise_slab_vst(x, 4, 30, 6, 9, model, vh, np.uint16(5), sigma=1.25)
        a = _args(fake, "b4d_denoise_slab_vst_u16")
        assert tuple(out.shape) == (3, 7, 8) and str(out.dtype).endswith("float32")
        assert a["out"] == (out.data_ptr() if isinstance(out, torch.Tensor) else out.ctypes.data)
        assert (a["z_begin"], a["z_total"], a["own_begin"], a["own_end"]) == (4, 30, 6, 9)
        assert a["first_value"] == 5 and type(a["first_value"]) is int and a["sigma_vst"] == 1.25
        assert (a["in_on_device"], a["out_on_device"]) == (False, False)
        pm = a["model"]._obj
        assert (pm.gain, pm.offset, pm.read_sigma) == (2.0, 37.0, 3.0)
        np.testing.assert_array_equal(fake.hists[-1], vh)
    q = d.denoise_slab_vst(slab, 0, 9, 0, 9, model, torch.from_numpy(vh), 5, quantize=(1.0, 2.0, 3.0, True))
    a = _args(fake, "b4d_denoise_slab_vst_q16_u16")
    assert q.dtype == np.uint16 and q.shape == slab.shape and a["out"] == q.ctypes.data
    assert (a["offset_sub"], a["offset_add"], a["step"], a["truncate"]) == (1.0, 2.0, 3.0, 1)
    d.slab_stage1_vst(slab, 2, 20, model, vh, 7, sigma=0.5)
    a = _args(fake, "b4d_slab_stage1_vst_u16")
    assert a["in"] == slab.ctypes.data and (a["z_begin"], a["z_total"], a["first_value"]) == (2, 20, 7)
    assert d._slab_shape == slab.shape
    n = len(fake.calls)
    for bad in (lambda: d.denoise_slab_vst(slab, 0, 9, 0, 9, model, vh[:100], 5),
                lambda: d.denoise_slab_vst(slab.astype(np.float32), 0, 9, 0, 9, model, vh, 5),
                lambda: d.slab_stage1_vst(slab, 0, 9, (0.0, 1.0, 1.0), vh, 5),
                lambda: d.denoise_slab_vst(slab, 0, 9, 0, 9, model, vh, 5, sigma=0.0)):
        with pytest.raises(ValueError):
            bad()
    assert len(fake.calls) == n


class _FakeShardDenoiser:
    """What the sharded orchestration calls: records the planes it counts and the slab calls."""

    def __init__(self, stages=2):
        import b4d

        self.profile, self._stages, self.calls = b4d.BM4DProfile(), stages, []

    def tile_stats(self, x, return_hist=False):
        self.calls.append(("tile_stats", np.array(x)))
        return {}, value_hist(x)

    def denoise_slab_vst(self, slab, z_begin, z_total, own_begin, own_end, model, vh, first, sigma=1.0):
        self.calls.append(("slab", z_begin, own_begin, own_end, model, np.array(vh), first, sigma))
        return np.zeros((own_end - own_begin,) + slab.shape[1:], np.float32)

    def slab_stage1_vst(self, slab, z_begin, z_total, model, vh, first, sigma=1.0):
        self.calls.append(("stage1", z_begin, model, np.array(vh), first, sigma))


def test_sharded_orchestration_merges_owned_plane_histograms(monkeypatch):
    from b4d import sharding
    from b4d.sharding import halo_planes, slab_plan

    rng = np.random.default_rng(48)
    vol = rng.integers(0, 4000, (90, 6, 8)).astype(np.uint16)
    merged = []

    def fake_merge(hist, group=None):
        merged.append(hist.numpy().copy())
        return hist * 3  # stands for the sum over the ranks

    monkeypatch.setattr(sharding, "merge_histograms", fake_merge)
    monkeypatch.setattr(sharding, "_process_group_ready", lambda: True)
    model = (2.0, 37.0, 3.0)
    for rank in range(3):
        d = _FakeShardDenoiser()
        ob, oe, out = sharding.denoise_volume_sharded(lambda a, b: vol[a:b], 90, 1.5, d, world=3, rank=rank,
                                                      model=model)
        want = slab_plan(90, 3, rank, halo_planes())
        assert (ob, oe) == want[:2] and out.shape == (oe - ob, 6, 8)
        (k0, planes), slab_call = d.calls
        assert k0 == "tile_stats"
        np.testing.assert_array_equal(planes, vol[ob:oe])
        np.testing.assert_array_equal(merged[-1], value_hist(vol[ob:oe]))
        _, zb, ob2, oe2, m, vh, first, sigma = slab_call
        assert (zb, ob2, oe2, m, first, sigma) == (want[2], ob, oe, model, int(vol[0, 0, 0]), 1.5)
        np.testing.assert_array_equal(vh, 3 * value_hist(vol[ob:oe]))
    # the exchange form takes the same value set and first voxel
    d = _FakeShardDenoiser()
    monkeypatch.setattr(sharding, "denoise_slab_exchange", lambda *a, **k: d.calls.append(("exchange", k)))
    sharding.denoise_volume_sharded(lambda a, b: vol[a:b], 90, 1.5, d, world=3, rank=1, exchange=True, model=model)
    assert d.calls[-1][1]["first"] == int(vol[0, 0, 0]) and d.calls[-1][1]["model"] == model


def test_sharded_vst_without_a_process_group_is_an_error():
    from b4d import sharding

    vol = np.ones((40, 6, 8), np.uint16)
    d = _FakeShardDenoiser()
    with pytest.raises(ValueError, match="process group"):
        sharding.denoise_volume_sharded(lambda a, b: vol[a:b], 40, 1.0, d, world=2, rank=0, model=(2.0, 0.0, 1.0))
    assert d.calls == []
    # a given value set needs no collective
    sharding.denoise_volume_sharded(lambda a, b: vol[a:b], 40, 1.0, d, world=2, rank=1, model=(2.0, 0.0, 1.0),
                                    value_hist=value_hist(vol))
    assert [c[0] for c in d.calls] == ["slab"]
    # one rank: its owned planes are the whole volume
    d = _FakeShardDenoiser()
    sharding.denoise_volume_sharded(lambda a, b: vol[a:b], 40, 1.0, d, world=1, rank=0, model=(2.0, 0.0, 1.0))
    np.testing.assert_array_equal(d.calls[-1][5], value_hist(vol))
