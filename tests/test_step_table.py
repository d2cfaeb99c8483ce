"""Per-tile quantizer steps (DESIGN §3 item 13): the standalone quantizer with a step table, its device inverse, and the
fused denoise -> quantize path with a table, whole, in slabs, in the two-call exchange form and pipelined.  A voxel's
result is what the scalar quantizer gives on it with its tile's step, bit for bit.  CPU tests: the header against the
binding's table, the Denoiser methods against a fake library, and the argument checks."""
import ctypes
import os

import numpy as np
import pytest

from test_binding import FakeLib, _prototypes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------- NumPy restatements ----
def per_voxel_steps(steps, tile, shape, z_begin=0):
    """The step of every voxel of planes [z_begin, z_begin + D) of the volume the table covers."""
    D, H, W = shape
    zi = (z_begin + np.arange(D)) // tile[0]
    return np.asarray(steps, np.float32)[np.ix_(zi, np.arange(H) // tile[1], np.arange(W) // tile[2])]


def quantize_numpy(x, s, sub=0.0, add=0.0, truncate=False):
    """K7 in float32 with a step per voxel (csrc/b4d_common.cuh quant1 / quant1_trunc)."""
    f32 = np.float32
    x, s = np.asarray(x, f32), np.asarray(s, f32)
    with np.errstate(invalid="ignore", over="ignore"):
        v = (x - f32(sub)).astype(f32) + f32(add)
        v = np.where(s == f32(1), v, (v / s).astype(f32)).astype(f32)
        v = np.where(np.isnan(v), f32(0), np.maximum(v, f32(0)))
        if truncate:
            return (np.trunc(v).astype(np.int64) & 0xFFFF).astype(np.uint16)
        hi = (f32(65535) / s).astype(f32)
        return np.rint(np.minimum(v, hi)).astype(np.uint16)


def dequantize_numpy(q, s, sub=0.0, add=0.0):
    f32 = np.float32
    return ((np.asarray(q).astype(f32) * np.asarray(s, f32)).astype(f32) + f32(sub) - f32(add)).astype(f32)


def ragged_table(seed=3):
    """(37, 41, 45) planes in (8, 16, 12) tiles: a 5 x 3 x 4 grid, ragged on every axis, with steps 1, 1.5, 3.7, 250."""
    import b4d

    rng = np.random.default_rng(seed)
    steps = rng.choice(np.array([1.0, 1.5, 3.7, 250.0, 2.0, 17.25], np.float32), (5, 3, 4))
    steps[0, 0, 0], steps[1, 1, 1], steps[2, 2, 2], steps[4, 2, 3] = 1.0, 1.5, 3.7, 250.0
    return b4d.StepTable(steps, (8, 16, 12))


def hard_input(shape, seed=4):
    """float32 with negatives, NaN, values far above every clip and values near the rounding midpoints."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-50.0, 2000.0, shape).astype(np.float32)
    flat = x.reshape(-1)
    n = flat.size
    flat[rng.choice(n, n // 50, replace=False)] = np.nan
    flat[rng.choice(n, n // 50, replace=False)] = rng.uniform(7.0e4, 3.0e7, n // 50).astype(np.float32)
    flat[rng.choice(n, n // 50, replace=False)] = rng.integers(0, 3000, n // 50).astype(np.float32) + 0.5
    flat[rng.choice(n, n // 50, replace=False)] = -rng.uniform(0.0, 1e6, n // 50).astype(np.float32)
    return x


def tiles_of(table, shape):
    tz, ty, tx = table.tile
    for iz in range(table.steps.shape[0]):
        for iy in range(table.steps.shape[1]):
            for ix in range(table.steps.shape[2]):
                sl = (slice(iz * tz, min((iz + 1) * tz, shape[0])), slice(iy * ty, (iy + 1) * ty),
                      slice(ix * tx, (ix + 1) * tx))
                if sl[0].start < shape[0]:
                    yield float(table.steps[iz, iy, ix]), sl


@pytest.fixture(scope="module")
def dn():
    import b4d

    d = b4d.Denoiser(0)
    yield d
    d.close()


# ---------------------------------------------------------------------------------------------------------- GPU --
@pytest.mark.gpu
@pytest.mark.parametrize("truncate", [False, True])
def test_tiled_quantize_equals_the_scalar_quantizer_per_tile(dn, truncate):
    import torch

    table = ragged_table()
    x = hard_input((37, 41, 45))
    for sub, add in ((0.0, 0.0), (37.0, 5.0)):
        got = dn.quantize(x, sub, add, table, truncate)
        np.testing.assert_array_equal(got, quantize_numpy(x, per_voxel_steps(table.steps, table.tile, x.shape), sub,
                                                          add, truncate))
        for s, sl in tiles_of(table, x.shape):
            np.testing.assert_array_equal(got[sl], dn.quantize(np.ascontiguousarray(x[sl]), sub, add, s, truncate))
        xt = torch.from_numpy(x).cuda()
        np.testing.assert_array_equal(dn.quantize(xt, sub, add, table, truncate).cpu().numpy(), got)
    # W % 4 == 0 and 16-byte aligned: the vector path
    x4 = hard_input((37, 41, 48), 5)
    t4 = ragged_table()._replace(tile=(8, 16, 12))
    np.testing.assert_array_equal(dn.quantize(x4, 1.0, 0.0, t4, truncate),
                                  quantize_numpy(x4, per_voxel_steps(t4.steps, t4.tile, x4.shape), 1.0, 0.0, truncate))


@pytest.mark.gpu
def test_plane_ranges_and_uniform_tables(dn):
    import b4d
    from b4d import synth

    table = ragged_table()
    x = hard_input((37, 41, 45), 6)
    whole = dn.quantize(x, 2.0, 1.0, table)
    for z0, z1 in ((10, 30), (8, 16), (33, 37)):
        np.testing.assert_array_equal(dn.quantize(np.ascontiguousarray(x[z0:z1]), 2.0, 1.0, table, z_begin=z0),
                                      whole[z0:z1])
    for s in (1.0, 2.5):
        uni = b4d.StepTable(np.full((5, 3, 4), s, np.float32), (8, 16, 12))
        for trunc in (False, True):
            np.testing.assert_array_equal(dn.quantize(x, 2.0, 1.0, uni, trunc), dn.quantize(x, 2.0, 1.0, s, trunc))
        v = synth.vol(37, 41, 45, seed=7)
        np.testing.assert_array_equal(dn.denoise_quantized(v, 24.0, 10.0, 0.0, uni),
                                      dn.denoise_quantized(v, 24.0, 10.0, 0.0, s))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(40, 44, 48), (37, 41, 45)])  # TMA normalise (W % 4 == 0) and the fallback
def test_fused_equals_quantize_of_denoise(dn, shape):
    import b4d
    from b4d import synth

    v = synth.vol(*shape, seed=8)
    y = dn.denoise(v, 24.0)
    for tile in ((8, 16, 12), (7, 5, 9)):
        grid = tuple(-(-n // t) for n, t in zip(shape, tile))
        steps = np.random.default_rng(9).choice(np.array([1.0, 1.5, 3.7, 250.0], np.float32), grid)
        table = b4d.StepTable(steps, tile)
        for sub, add, trunc in ((0.0, 0.0, False), (40.0, 3.0, False), (40.0, 3.0, True)):
            np.testing.assert_array_equal(dn.denoise_quantized(v, 24.0, sub, add, table, trunc),
                                          dn.quantize(y, sub, add, table, trunc))


def _slab_case():
    import b4d
    from b4d import synth

    v = synth.vol(90, 24, 28, seed=10)
    steps = np.random.default_rng(11).choice(np.array([1.0, 1.5, 3.7, 250.0], np.float32), (13, 3, 4))
    return v, b4d.StepTable(steps, (7, 10, 9))  # tile layers end at 7k: no slab boundary is aligned to them


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_slabs_concatenate_to_the_whole_volume(dn, world):
    import torch

    import b4d
    from b4d.sharding import exchange_halo, halo_planes, slab_plan

    v, table = _slab_case()
    D = v.shape[0]
    for q in ((37.0, 0.0, table), (37.0, 5.0, table, True)):
        whole = dn.denoise_quantized(v, 24.0, *q)
        parts, tparts = [], []
        for r in range(world):
            ob, oe, zb, ze = slab_plan(D, world, r, halo_planes())
            parts.append(dn.denoise_slab(v[zb:ze], zb, D, ob, oe, 24.0, quantize=q))
            vt = torch.from_numpy(v[zb:ze].view(np.int16)).view(torch.uint16).cuda()
            tparts.append(dn.denoise_slab(vt, zb, D, ob, oe, 24.0, quantize=q).cpu().numpy())
        np.testing.assert_array_equal(np.concatenate(parts, 0), whole)
        np.testing.assert_array_equal(np.concatenate(tparts, 0), whole)
        # the two-call form with one exchange of basic-estimate planes (staging copies)
        h = exchange_halo(11, 11)
        ranks = []
        for r in range(world):
            ob, oe, zb, ze = slab_plan(D, world, r, h)
            d = b4d.Denoiser(0)
            d.slab_stage1(v[zb:ze], zb, D, 24.0)
            ranks.append((d, ob, oe, zb, ze))
        sends = [(d.slab_basic(ob - zb, h), d.slab_basic(oe - zb - h, h)) for d, ob, oe, zb, ze in ranks]
        parts = []
        for r, (d, ob, oe, zb, ze) in enumerate(ranks):
            if r > 0:
                d.slab_set_basic(0, sends[r - 1][1])
            if r < world - 1:
                d.slab_set_basic(oe - zb, sends[r + 1][0])
            out = d.slab_stage2(ob, oe, quantize=q) if r % 2 == 0 else d.slab_stage2(
                ob, oe, device=torch.device("cuda", 0), quantize=q).cpu().numpy()
            parts.append(out)
            d.close()
        np.testing.assert_array_equal(np.concatenate(parts, 0), whole)


@pytest.mark.gpu
def test_pipelined_host_output_equals_device_output():
    import torch

    import b4d
    from b4d import synth

    v = synth.vol(208, 16, 20, seed=12)
    steps = np.random.default_rng(13).choice(np.array([1.0, 1.5, 3.7, 250.0], np.float32), (30, 2, 3))
    table = b4d.StepTable(steps, (7, 9, 8))
    d = b4d.Denoiser(0)
    try:
        d.set_pipeline_min_voxels(0)
        vt = torch.from_numpy(v.view(np.int16)).view(torch.uint16).cuda()
        for trunc in (False, True):
            dev_out = d.denoise_slab(vt, 0, 208, 0, 208, 24.0, quantize=(37.0, 0.0, table, trunc)).cpu().numpy()
            host = d.denoise_quantized(v, 24.0, 37.0, 0.0, table, trunc)
            assert d.last_timings()["norm2"][1] > 1  # the chunked normalise ran
            np.testing.assert_array_equal(host, dev_out)
            np.testing.assert_array_equal(dev_out, d.quantize(d.denoise(vt, 24.0), 37.0, 0.0, table, trunc)
                                          .cpu().numpy())
    finally:
        d.close()


@pytest.mark.gpu
def test_dequantize_and_the_round_trip(dn):
    import torch

    import b4d

    table = ragged_table()
    s = per_voxel_steps(table.steps, table.tile, (37, 41, 45))
    q = np.random.default_rng(14).integers(0, 65536, (37, 41, 45)).astype(np.uint16)
    for sub, add in ((0.0, 0.0), (37.5, 3.25)):
        np.testing.assert_array_equal(dn.dequantize(q, table, sub, add), dequantize_numpy(q, s, sub, add))
        qt = torch.from_numpy(q.view(np.int16)).view(torch.uint16).cuda()
        np.testing.assert_array_equal(dn.dequantize(qt, table, sub, add).cpu().numpy(), dequantize_numpy(q, s, sub, add))
    np.testing.assert_array_equal(dn.dequantize(q[:, :, :44], 2.5, 1.0), dequantize_numpy(q[:, :, :44], 2.5, 1.0))
    np.testing.assert_array_equal(dn.dequantize(np.ascontiguousarray(q[9:20]), table, z_begin=9),
                                  dequantize_numpy(q[9:20], s[9:20]))
    np.testing.assert_array_equal(b4d.dequantize(q, table), dequantize_numpy(q, s))
    # inside the clip range of the rounding quantizer the round trip is within half a step
    x = np.random.default_rng(15).uniform(30.0, 60000.0, (37, 41, 45)).astype(np.float32)
    xh = dn.dequantize(dn.quantize(x, 30.0, 0.0, table), table, 30.0, 0.0)
    assert np.all(np.abs(xh.astype(np.float64) - x) <= s / 2 + 4 * np.spacing(np.float32(60000.0)))


def _launches(d):
    return sum(n for _, n in d.last_timings().values())


def _profiled_kernels(call, tmp_path):
    """Kernels the CUDA profiler records during `call` (memcpy and memset excluded), after one warm-up call."""
    import json

    import torch

    call()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    trace = os.path.join(str(tmp_path), "trace.json")
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    return sum(1 for e in events if e.get("cat") == "kernel")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fused", "two_call_begin"])
def test_booked_launches_equal_the_profiler(name, tmp_path):
    import b4d
    from b4d import synth

    d = b4d.Denoiser(0)
    v = synth.vol(64, 64, 64, seed=16)
    table = b4d.StepTable(np.random.default_rng(17).choice(np.array([1.0, 3.7], np.float32), (10, 5, 6)), (7, 13, 11))
    if name == "fused":
        call = lambda: d.denoise_quantized(v, 24.0, 10.0, 0.0, table)  # noqa: E731
    else:
        def call():
            d.slab_stage1(v[8:56], 8, 64, 24.0)
            d.slab_stage2_begin(16, 48)
            d.slab_stage2(16, 48, quantize=(10.0, 0.0, table))
    try:
        kernels = _profiled_kernels(call, tmp_path)
        assert _launches(d) == kernels, (kernels, d.last_timings())
    finally:
        d.close()


@pytest.mark.gpu
def test_noise_scaled_steps_follow_the_noise(dn):
    import b4d

    rng = np.random.default_rng(18)
    shape = (48, 32, 64)
    z, y, x = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    clean = 1000.0 + 300.0 * np.sin(z / 5.0) * np.cos(y / 7.0) + 2.0 * x
    noise = rng.normal(0.0, 1.0, shape) * np.where(x < 32, 8.0, 32.0)
    v = np.clip(np.rint(clean + noise), 0, 65535).astype(np.uint16)
    tile = (16, 16, 16)
    table = b4d.noise_scaled_steps(dn.noise_sigma(v, tile=tile)["sigma"], 0.5, tile)
    left, right = table.steps[:, :, :2], table.steps[:, :, 2:]
    assert left.max() < 6.0 and right.min() > 12.0, table.steps
    got = dn.denoise_quantized(v, 20.0, 900.0, 0.0, table)
    by_step = {}
    for s, sl in tiles_of(table, shape):
        if s not in by_step:
            by_step[s] = dn.denoise_quantized(v, 20.0, 900.0, 0.0, s)
        np.testing.assert_array_equal(got[sl], by_step[s][sl])


# ---------------------------------------------------------------------------------------------------------- CPU --
STEP_PROTOS = _prototypes("b4d_step_table.h")
STEP_PARAMS = {name: [n for _, n in params] for name, (_, params) in STEP_PROTOS.items()}


def test_header_matches_the_table():
    from b4d import _lib

    scalars = {"int64_t": ctypes.c_int64, "int": ctypes.c_int, "float": ctypes.c_float, "double": ctypes.c_double}
    assert sorted(_lib.STEP_TABLE_EXPORTS) == sorted(STEP_PROTOS) and len(STEP_PROTOS) == 4
    for name, (ret, params) in STEP_PROTOS.items():
        restype, argtypes = _lib.STEP_TABLE_SIGNATURES[name]
        assert ret == "int" and restype is ctypes.c_int
        assert argtypes == [ctypes.c_void_p if t == "*" else scalars[t] for t, _ in params], name
    assert not set(_lib.STEP_TABLE_SIGNATURES) & (set(_lib.SIGNATURES) | set(_lib.VST_SLAB_SIGNATURES))


def _fake_denoiser():
    import b4d
    from b4d import _lib

    fake = FakeLib()
    for name, (_, argtypes) in {**_lib.VST_SLAB_SIGNATURES, **_lib.STEP_TABLE_SIGNATURES}.items():
        setattr(fake, name, fake._fn(name, argtypes, 0))
    d = object.__new__(b4d.Denoiser)
    d.lib, d.device, d.profile, d._stages = fake, 0, b4d.BM4DProfile(), 2
    d._h, d._pid = ctypes.c_void_p(0x1000), os.getpid()
    return d, fake


def _args(fake, name):
    called, args = fake.calls[-1]
    assert called == name
    return dict(zip(STEP_PARAMS[name], args))


def _table_args(a, table):
    """(tile, grid, steps) a call received."""
    grid = tuple(a["grid"])
    steps = np.ctypeslib.as_array((ctypes.c_float * int(np.prod(grid))).from_address(a["steps"])).reshape(grid)
    return tuple(a["tile"]), grid, steps


def test_denoiser_methods_on_a_fake_library():
    import torch

    import b4d

    d, fake = _fake_denoiser()
    table = ragged_table()
    x = np.zeros((37, 41, 45), np.float32)
    for xx in (x, torch.from_numpy(x)):
        out = d.quantize(xx, 1.5, 2.5, table, True)
        a = _args(fake, "b4d_quantize_tiled_u16")
        assert tuple(out.shape) == x.shape and str(out.dtype).endswith("uint16")
        assert a["in"] == (xx.data_ptr() if isinstance(xx, torch.Tensor) else x.ctypes.data)
        assert a["out"] == (out.data_ptr() if isinstance(out, torch.Tensor) else out.ctypes.data)
        assert (tuple(a["shape"]), a["z_begin"], a["offset_sub"], a["offset_add"], a["truncate"]) == (
            (37, 41, 45), 0, 1.5, 2.5, 1)
        assert (a["in_on_device"], a["out_on_device"]) == (False, False)
        tile, grid, steps = _table_args(a, table)
        assert tile == (8, 16, 12) and grid == (5, 3, 4)
        np.testing.assert_array_equal(steps, table.steps)
    d.quantize(np.ascontiguousarray(x[20:30]), 0, 0, table, z_begin=20)
    a = _args(fake, "b4d_quantize_tiled_u16")
    assert a["z_begin"] == 20 and tuple(a["shape"]) == (10, 41, 45) and a["truncate"] == 0
    # scalar steps reach the scalar symbols with the arguments they always had
    out = d.quantize(x, 1.5, 2.5, 3.0)
    assert fake.calls[-1] == ("b4d_quantize_u16", (d._h, x.ctypes.data, x.size, 1.5, 2.5, 3.0, out.ctypes.data,
                                                   False, False))
    d.quantize(x, 1.5, 2.5, 3.0, True)
    assert fake.calls[-1][0] == "b4d_quantize_trunc_u16"
    # dequantize: a scalar is a one-tile table
    q = np.zeros((9, 7, 8), np.uint16)
    out = d.dequantize(q, 2.5, 1.0, 0.5, z_begin=3)
    a = _args(fake, "b4d_dequantize_tiled_f32")
    assert out.dtype == np.float32 and a["out"] == out.ctypes.data and a["in"] == q.ctypes.data
    tile, grid, steps = _table_args(a, None)
    assert tile == (12, 7, 8) and grid == (1, 1, 1) and steps.ravel().tolist() == [2.5]
    assert (a["z_begin"], a["offset_sub"], a["offset_add"]) == (3, 1.0, 0.5)
    t2 = b4d.StepTable(np.full((2, 1, 1), 4.0, np.float32), (5, 7, 8))
    d.dequantize(q, t2)
    assert _table_args(_args(fake, "b4d_dequantize_tiled_f32"), t2)[:2] == ((5, 7, 8), (2, 1, 1))
    # the fused path: slabs, the whole volume, the two-call form
    slab = np.zeros((30, 41, 45), np.uint16)
    out = d.denoise_slab(slab, 5, 37, 10, 30, 24.0, quantize=(3.0, 1.0, table, True))
    a = _args(fake, "b4d_denoise_slab_qt16_u16")
    assert out.shape == (20, 41, 45) and out.dtype == np.uint16 and a["out"] == out.ctypes.data
    assert (a["z_begin"], a["z_total"], a["own_begin"], a["own_end"], a["sigma"]) == (5, 37, 10, 30, 24.0)
    assert (a["offset_sub"], a["offset_add"], a["truncate"]) == (3.0, 1.0, 1)
    assert _table_args(a, table)[:2] == ((8, 16, 12), (5, 3, 4))
    vol = np.zeros((37, 41, 45), np.uint16)
    d.denoise_quantized(vol, 24.0, 3.0, 0.0, table)
    a = _args(fake, "b4d_denoise_slab_qt16_u16")
    assert (a["z_begin"], a["z_total"], a["own_begin"], a["own_end"], a["truncate"]) == (0, 37, 0, 37, 0)
    out = d.denoise_quantized(vol, 24.0, 3.0, 0.0, 2.0)
    assert fake.calls[-1][0] == "b4d_denoise_slab_q16_u16" and fake.calls[-1][1][8:12] == (3.0, 0.0, 2.0, 0)
    d.slab_stage1(slab, 5, 37, 24.0)
    out = d.slab_stage2(10, 30, quantize=(3.0, 1.0, table))
    a = _args(fake, "b4d_slab_stage2_qt16")
    assert (a["own_begin"], a["own_end"], a["offset_sub"], a["offset_add"], a["truncate"]) == (10, 30, 3.0, 1.0, 0)
    assert a["out"] == out.ctypes.data and a["out_on_device"] is False
    assert _table_args(a, table)[:2] == ((8, 16, 12), (5, 3, 4))
    d.slab_stage2(10, 30, quantize=(3.0, 1.0, 2.0))
    assert fake.calls[-1][0] == "b4d_slab_stage2_q16" and fake.calls[-1][1][3:7] == (3.0, 1.0, 2.0, 0)


def test_module_level_calls_and_the_exchange_form(monkeypatch):
    import b4d
    from b4d import api, sharding

    d, fake = _fake_denoiser()
    monkeypatch.setattr(api, "get_denoiser", lambda device=None: d)
    table = ragged_table()
    b4d.quantize(np.zeros((37, 41, 45), np.float32), 1.0, 0.0, table, truncate=True)
    assert _args(fake, "b4d_quantize_tiled_u16")["truncate"] == 1
    b4d.dequantize(np.zeros((37, 41, 45), np.uint16), table, 1.0)
    assert _args(fake, "b4d_dequantize_tiled_f32")["offset_sub"] == 1.0
    b4d.denoise_quantized(np.zeros((37, 41, 45), np.uint16), 24.0, 0.0, 0.0, table)
    assert _args(fake, "b4d_denoise_slab_qt16_u16")["z_total"] == 37
    slab = np.zeros((37, 41, 45), np.uint16)
    out = sharding.denoise_slab_exchange(d, slab, 0, 37, 0, 37, 24.0, 0, 1, quantize=(2.0, 0.0, table))
    assert [c for c, _ in fake.calls[-2:]] == ["b4d_slab_stage1_u16", "b4d_slab_stage2_qt16"]
    assert out.shape == (37, 41, 45) and out.dtype == np.uint16
    n = len(fake.calls)
    with pytest.raises(ValueError):
        sharding.denoise_slab_exchange(d, slab, 0, 48, 0, 37, 24.0, 0, 1, quantize=(2.0, 0.0, table))
    with pytest.raises(NotImplementedError):
        sharding.denoise_slab_exchange(d, slab, 0, 37, 0, 37, 1.0, 0, 1, quantize=(2.0, 0.0, table),
                                       model=(2.0, 0.0, 1.0), value_hist=np.ones(65536, np.int64), first=0)
    assert len(fake.calls) == n


def test_bad_tables_raise_before_the_library():
    import b4d

    d, fake = _fake_denoiser()
    x = np.zeros((37, 41, 45), np.float32)
    vol = np.zeros((37, 41, 45), np.uint16)
    good = ragged_table()

    def with_step(i, v):
        s = good.steps.copy()
        s.reshape(-1)[i] = v
        return b4d.StepTable(s, good.tile)

    bad_tables = [with_step(3, np.nan), with_step(5, np.inf), with_step(7, -np.inf), with_step(0, 0.5),
                  b4d.StepTable(good.steps[0], good.tile[1:] + (1,)),   # 2-D
                  b4d.StepTable(good.steps[:, :2], good.tile),          # nty does not match H
                  b4d.StepTable(good.steps[:, :, :3], good.tile),       # ntx does not match W
                  b4d.StepTable(good.steps, (8, 16, 11)),               # ntx does not match W in tiles of 11
                  b4d.StepTable(good.steps[:4], good.tile),             # planes beyond the grid
                  b4d.StepTable(good.steps, (0, 16, 12))]               # tile side < 1
    n = len(fake.calls)
    for t in bad_tables:
        for call in (lambda: d.quantize(x, 0.0, 0.0, t), lambda: d.dequantize(vol, t),
                     lambda: d.denoise_quantized(vol, 24.0, 0.0, 0.0, t),
                     lambda: d.denoise_slab(vol[:30], 5, 37, 10, 30, 24.0, quantize=(0.0, 0.0, t))):
            with pytest.raises(ValueError):
                call()
    # z_begin beyond the grid, and a slab table that does not cover exactly z_total planes
    for call in (lambda: d.quantize(np.ascontiguousarray(x[:10]), 0.0, 0.0, good, z_begin=31),
                 lambda: d.dequantize(vol[:10], good, z_begin=31), lambda: d.quantize(x, 0.0, 0.0, good, z_begin=-1),
                 lambda: d.denoise_slab(vol[:30], 0, 30, 0, 30, 24.0, quantize=(0.0, 0.0, good)),
                 lambda: d.dequantize(vol, 0.5), lambda: b4d.quantize(x[:, :, :30], 0.0, 0.0, good),
                 lambda: b4d.dequantize(vol, good._replace(steps=good.steps[:, :, :2]))):
        with pytest.raises(ValueError):
            call()
    d.slab_stage1(vol, 0, 37, 24.0)
    with pytest.raises(ValueError):
        d.slab_stage2(0, 37, quantize=(0.0, 0.0, good._replace(steps=good.steps[:4])))
    assert [c for c, _ in fake.calls[n:]] == ["b4d_slab_stage1_u16"]


def test_a_table_on_the_vst_path_is_not_implemented():
    import b4d

    d, fake = _fake_denoiser()
    vol = np.zeros((37, 41, 45), np.uint16)
    m, vh = b4d.PoissonGaussian(2.0, 37.0, 3.0), np.ones(65536, np.int64)
    q = (0.0, 0.0, ragged_table())
    for call in (lambda: d.denoise_vst(vol, m, quantize=q), lambda: b4d.denoise_vst(vol, m, quantize=q),
                 lambda: d.denoise_slab_vst(vol, 0, 37, 0, 37, m, vh, 0, quantize=q)):
        with pytest.raises(NotImplementedError):
            call()
    assert fake.calls == []
    d.slab_stage1_vst(vol, 0, 37, m, vh, 0)
    with pytest.raises(NotImplementedError):
        d.slab_stage2(0, 37, quantize=q)
    assert [c for c, _ in fake.calls] == ["b4d_slab_stage1_vst_u16"]


def test_noise_scaled_steps_match_noise_scaled_step():
    import torch

    import b4d

    sigma = np.array([[[np.nan, 0.0, 1.0], [2.0, 7.3, 24.0]], [[1e-9, 3.3e3, np.nan], [0.5, 1.999, 2.001]]])
    for kappa in (0.5, 1.0, 3.7):
        for s in (sigma, torch.from_numpy(sigma)):
            t = b4d.noise_scaled_steps(s, kappa, (64, 32, 16))
            assert isinstance(t, b4d.StepTable) and t.tile == (64, 32, 16) and t.steps.dtype == np.float32
            want = [1.0 if np.isnan(v) else np.float32(b4d.noise_scaled_step(v, kappa)) for v in sigma.ravel()]
            np.testing.assert_array_equal(t.steps.ravel(), np.array(want, np.float32))
