"""The ctypes binding: the signature table of b4d/_lib.py against the prototypes of both headers, every Denoiser
method against a fake library that converts each argument through its prototype (pointers, on-device flags, returned
kinds), and the refusal of CUDA tensors and outputs on a device other than the handle's."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADERS = {"b4d.h": "EXPORTS", "b4d_noise.h": "NOISE_EXPORTS"}
SCALARS = {"int64_t": ctypes.c_int64, "int": ctypes.c_int, "float": ctypes.c_float, "double": ctypes.c_double}


def _prototypes(header):
    """name -> (return type, [(parameter type, parameter name)]) of every function the header declares."""
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", header)).read(), flags=re.S)
    protos = {}
    for ret, name, params in re.findall(r"^((?:const\s+)?\w+[\s*]+?)\s*(b4d_\w+)\s*\(([^)]*)\)\s*;", src, flags=re.M):
        parsed = []
        for p in params.split(","):
            p = " ".join(p.split())
            if p and p != "void":
                m = re.match(r"(.*?)\s*\**\s*(\w+)(\[\w*\])?$", p)
                ptr = "*" in p or m.group(3) is not None
                parsed.append(("*" if ptr else m.group(1).replace("const ", ""), m.group(2)))
        protos[name] = (" ".join(ret.split()), parsed)
    return protos


def _mapped_restype(ret):
    if ret == "void":
        return None
    if ret == "const char *":
        return ctypes.c_char_p
    return ctypes.c_void_p if ret.endswith("*") else SCALARS[ret]


PROTOS = {name: p for h in HEADERS for name, p in _prototypes(h).items()}
PARAMS = {name: [n for _, n in params] for name, (_, params) in PROTOS.items()}


# ------------------------------------------------------ header <-> table ----
def test_table_matches_the_headers():
    from b4d import _lib

    assert len(PROTOS) == 42
    for header, exports in HEADERS.items():
        declared = _prototypes(header)
        assert sorted(getattr(_lib, exports)) == sorted(declared), header
        for name, (ret, params) in declared.items():
            restype, argtypes = _lib.SIGNATURES[name]
            assert restype is _mapped_restype(ret), name
            want = [ctypes.c_void_p if t == "*" else SCALARS[t] for t, _ in params]
            assert len(argtypes) == len(want) and all(a is w for a, w in zip(argtypes, want)), name
    assert sorted(_lib.SIGNATURES) == sorted(PROTOS)


@pytest.fixture(scope="module")
def lib():
    from b4d import _lib

    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return _lib.load()


def test_load_applies_the_table(lib):
    from b4d import _lib

    for name, (restype, argtypes) in _lib.SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


# ------------------------------------------------- methods on a fake library ----
class FakeLib:
    """One callable per table entry: checks the arity, converts every argument with its argtype's from_param (an
    ndarray in a pointer slot, a float in an integer slot ... raise), records the call and returns 0."""

    def __init__(self, returns=None):
        from b4d import _lib

        self.calls = []
        for name, (_, argtypes) in _lib.SIGNATURES.items():
            setattr(self, name, self._fn(name, argtypes, (returns or {}).get(name, 0)))

    def _fn(self, name, argtypes, ret):
        def call(*args):
            assert len(args) == len(argtypes), "%s takes %d arguments, got %d" % (name, len(argtypes), len(args))
            for t, v in zip(argtypes, args):
                t.from_param(v)
            self.calls.append((name, args))
            return ret

        return call

    def last(self, name):
        """Arguments of the last call, by the header's parameter names; it must have been a call of `name`."""
        called, args = self.calls[-1]
        assert called == name
        return dict(zip(PARAMS[name], args))


R_REFS = 5  # what the fake's b4d_num_refs returns


def _denoiser(fake, device=0):
    import b4d

    d = object.__new__(b4d.Denoiser)
    d.lib, d.device, d.profile, d._stages = fake, device, b4d.BM4DProfile(), 2
    d._h, d._pid = ctypes.c_void_p(0x1000), os.getpid()
    return d


@pytest.fixture()
def fake():
    return FakeLib({"b4d_num_refs": R_REFS})


def _addr(a):
    return a.data_ptr() if type(a).__module__.startswith("torch") else a.ctypes.data


def _host_flags(args):
    return [v for k, v in args.items() if k.endswith("on_device")]


def _kinds(x):
    """The array kinds a method is run with: NumPy, and a CPU tensor sharing its memory."""
    import torch

    return [x, torch.from_numpy(x)]


def _same_kind(out, x, shape, dtype):
    import torch

    if isinstance(x, torch.Tensor):
        assert isinstance(out, torch.Tensor) and out.device.type == "cpu" and out.dtype == getattr(torch, dtype)
    else:
        assert isinstance(out, np.ndarray) and out.dtype == dtype
    assert tuple(out.shape) == tuple(shape)


VOL = np.arange(6 * 7 * 8, dtype=np.uint16).reshape(6, 7, 8)


def test_denoise_and_denoise_ptr(fake):
    d = _denoiser(fake)
    for x, fn in ((VOL, "b4d_denoise_u16"), (VOL.astype(np.float32)[None].repeat(2, 0), "b4d_denoise_f32")):
        for xi in _kinds(x):
            y = d.denoise(xi, 24.0)
            a = fake.last(fn)
            _same_kind(y, xi, x.shape, "float32")
            assert a["in"] == _addr(xi) and a["out"] == _addr(y) and _host_flags(a) == [0, 0]
            assert a["n"] == (1 if x.ndim == 3 else 2) and list(a["shape"]) == list(x.shape[-3:]) and a["sigma"] == 24
    d.denoise_ptr(0x2000, np.uint16, 3, (4, 5, 6), 10.0, 0x3000, False, False)
    a = fake.last("b4d_denoise_u16")
    assert (a["in"], a["n"], list(a["shape"]), a["out"]) == (0x2000, 3, [4, 5, 6], 0x3000)


def test_targets_and_foreground_mask(fake):
    d = _denoiser(fake)
    x = np.stack([VOL, VOL])
    raw, teacher = d.targets(x, [1.0, 2.0], 24.0)
    a = fake.last("b4d_targets_u16")
    for o in (raw, teacher):
        _same_kind(o, x, x.shape, "float32")
    assert (a["in"], a["raw_out"], a["teacher_out"]) == (x.ctypes.data, raw.ctypes.data, teacher.ctypes.data)
    assert a["n"] == 2 and _host_flags(a) == [0, 0]
    mine = np.empty(x.shape, np.float32)
    assert d.targets(x, 0.0, 24.0, raw_out=mine)[0] is mine
    assert fake.last("b4d_targets_u16")["raw_out"] == mine.ctypes.data
    with pytest.raises(ValueError):
        d.targets(x, 0.0, 24.0, teacher_out=np.empty(x.shape, np.float64))
    for xi, n in ((VOL, 1), (x, 2)):
        m = d.foreground_mask(xi, 3.0)
        a = fake.last("b4d_foreground_mask_u16")
        _same_kind(m, xi, xi.shape, "bool")
        assert (a["in"], a["out"], a["n"], a["dilate"]) == (xi.ctypes.data, m.ctypes.data, n, 1)
        assert _host_flags(a) == [0, 0]


def test_slab_calls(fake):
    d = _denoiser(fake)
    ob, oe = 1, 4
    for xi in _kinds(VOL):
        for quant, fn, dt in ((None, "b4d_denoise_slab_u16", "float32"),
                              ((2.0, 1.0, 3.0), "b4d_denoise_slab_q16_u16", "uint16")):
            y = d.denoise_slab(xi, 10, 40, 10 + ob, 10 + oe, 24.0, quantize=quant)
            a = fake.last(fn)
            _same_kind(y, xi, (oe - ob, 7, 8), dt)
            assert a["in"] == _addr(xi) and a["out"] == _addr(y) and _host_flags(a) == [0, 0]
            assert (a["z_begin"], a["z_total"], a["own_begin"], a["own_end"]) == (10, 40, 11, 14)
            if quant is not None:
                assert (a["offset_sub"], a["offset_add"], a["step"], a["truncate"]) == (2.0, 1.0, 3.0, 0)
        q = d.denoise_quantized(xi, 24.0, 1.0, 0.0, 2.0, truncate=True)
        a = fake.last("b4d_denoise_slab_q16_u16")
        _same_kind(q, xi, VOL.shape, "uint16")
        assert a["truncate"] == 1 and a["out"] == _addr(q)
        d.slab_stage1(xi, 10, 40, 24.0)
        a = fake.last("b4d_slab_stage1_u16")
        assert a["in"] == _addr(xi) and list(a["shape"]) == [6, 7, 8] and _host_flags(a) == [0]
    pinned = np.empty((oe - ob, 7, 8), np.float32)
    assert d.denoise_slab(VOL, 10, 40, 11, 14, 24.0, out=pinned) is pinned
    assert fake.last("b4d_denoise_slab_u16")["out"] == pinned.ctypes.data
    with pytest.raises(ValueError):
        d.denoise_slab(VOL, 10, 40, 11, 14, 24.0, out=np.empty((oe - ob, 7, 9), np.float32))

    basic = d.slab_basic(2, 3)
    a = fake.last("b4d_slab_basic_planes")
    _same_kind(basic, VOL, (3, 7, 8), "float32")
    assert (a["plane0"], a["nplanes"], a["buf"], a["to_handle"], a["buf_on_device"]) == (2, 3, basic.ctypes.data, 0, 0)
    planes = np.ones((2, 7, 8), np.float32)
    for pi in _kinds(planes):
        d.slab_set_basic(5, pi)
        a = fake.last("b4d_slab_basic_planes")
        assert (a["plane0"], a["nplanes"], a["buf"], a["to_handle"], a["buf_on_device"]) == (5, 2, _addr(pi), 1, 0)
    d.slab_set_basic(0, planes.astype(np.float64))  # NumPy planes are cast to float32
    with pytest.raises(ValueError):
        d.slab_set_basic(0, np.ones((2, 7, 9), np.float32))
    d.slab_stage2_begin(11, 14)
    assert fake.last("b4d_slab_stage2_begin") == {"h": d._h, "own_begin": 11, "own_end": 14}
    for quant, fn, dt in ((None, "b4d_slab_stage2", "float32"),
                          ((2.0, 1.0, 3.0, True), "b4d_slab_stage2_q16", "uint16")):
        y = d.slab_stage2(11, 14, quantize=quant)
        a = fake.last(fn)
        _same_kind(y, VOL, (3, 7, 8), dt)
        assert (a["own_begin"], a["own_end"], a["out"], a["out_on_device"]) == (11, 14, y.ctypes.data, 0)
    assert d.slab_stage2(11, 14, out=pinned) is pinned and fake.last("b4d_slab_stage2")["out"] == pinned.ctypes.data


def test_match_stage1(fake):
    d = _denoiser(fake)
    idx, ssd, cnt = d.match_stage1(VOL, 24.0)
    a = fake.last("b4d_match_stage1")
    K = d.profile.max_stack_size_ht
    assert (idx.shape, idx.dtype, ssd.shape, ssd.dtype, cnt.shape, cnt.dtype) == (
        (R_REFS, K), np.int32, (R_REFS, K), np.uint64, (R_REFS,), np.int32)
    assert (a["in"], a["idx"], a["ssd"], a["count"]) == (VOL.ctypes.data, idx.ctypes.data, ssd.ctypes.data,
                                                         cnt.ctypes.data)


def test_quantize_chunk_shuffle_tile_stats(fake):
    import torch

    d = _denoiser(fake)
    x = np.linspace(0, 9, 6 * 7 * 8, dtype=np.float32).reshape(6, 7, 8)
    for xi in _kinds(x):
        for trunc, fn in ((False, "b4d_quantize_u16"), (True, "b4d_quantize_trunc_u16")):
            q = d.quantize(xi, 1.0, 2.0, 3.0, truncate=trunc)
            a = fake.last(fn)
            _same_kind(q, xi, x.shape, "uint16")
            assert (a["in"], a["out"], a["n"], a["step"]) == (_addr(xi), _addr(q), x.size, 3.0)
            assert _host_flags(a) == [0, 0]
    q = d.quantize(x.astype(np.float64))  # NumPy input is cast to float32
    _same_kind(q, x, x.shape, "uint16")

    for xi in _kinds(VOL):
        out, hist = d.chunk_shuffle(xi, (4, 4, 4))
        a = fake.last("b4d_chunk_shuffle_u16")
        _same_kind(out, xi, (2 * VOL.size,), "uint8")
        _same_kind(hist, xi, (8, 2, 256), "int32" if isinstance(xi, torch.Tensor) else "uint32")
        assert (a["in"], a["out"], a["hist"]) == (_addr(xi), _addr(out), _addr(hist)) and _host_flags(a) == [0, 0]
        assert list(a["chunk"]) == [4, 4, 4]
        out, hist = d.chunk_shuffle(xi, want_hist=False)
        assert hist is None and fake.last("b4d_chunk_shuffle_u16")["hist"] is None

        st = d.tile_stats(xi, 2.0)
        a = fake.last("b4d_tile_stats")
        assert set(st) == {"n", "n_nonzero", "offset", "median", "mad", "sigma", "vmin", "vmax"}
        assert (a["in"], a["n"], a["pct"], a["hist"], a["in_on_device"]) == (_addr(xi), VOL.size, 2.0, None, 0)
        st, hist = d.tile_stats(xi, return_hist=True)
        assert isinstance(hist, np.ndarray) and hist.shape == (65536,) and hist.dtype == np.int64
        assert fake.last("b4d_tile_stats")["hist"] == hist.ctypes.data


def test_noise_and_vst(fake):
    import b4d

    d = _denoiser(fake)
    x = np.stack([VOL, VOL])
    model = b4d.PoissonGaussian(2.0, 10.0, 1.0)
    for xi in _kinds(x):
        r, hist = d.noise_sigma(xi, tile=(4, 4, 4), return_hist=True)
        a = fake.last("b4d_noise_sigma_u16")
        assert {k: (v.shape, v.dtype) for k, v in r.items()} == {"sigma": ((2, 2, 2, 2), np.float64),
                                                                 "mad": ((2, 2, 2, 2), np.float64),
                                                                 "cells": ((2, 2, 2, 2), np.int64)}
        assert (a["in"], a["n"], list(a["tile"]), a["sigma"], a["mad"], a["cells"], a["hist"], a["in_on_device"]) == (
            _addr(xi), 2, [4, 4, 4], r["sigma"].ctypes.data, r["mad"].ctypes.data, r["cells"].ctypes.data,
            hist.ctypes.data, 0)
        assert hist.shape == (262141,) and hist.dtype == np.int64
        r = d.noise_sigma(xi[0])
        assert np.shape(r["sigma"]) == () and fake.last("b4d_noise_sigma_u16")["tile"] is None

        f = d.noise_level_function(xi, edges=[0.0, 10.0, 100.0], min_cells=3)
        a = fake.last("b4d_noise_level_u16")
        assert (a["in"], a["n"], a["nbins"], a["min_cells"], a["edges"], a["cells"], a["in_on_device"]) == (
            _addr(xi), 2, 2, 3, f["edges"].ctypes.data, f["cells"].ctypes.data, 0)
        assert all(f[k].shape == (2,) for k in ("cells", "level_sum", "level", "mad", "sigma"))
        assert f["cells"].dtype == np.int64 and f["level"].dtype == np.float64 and isinstance(f["usable"], int)

        y = d.gat_forward(xi, model)
        a = fake.last("b4d_gat_forward_u16")
        _same_kind(y, xi, x.shape, "float32")
        assert (a["in"], a["out"], a["n"]) == (_addr(xi), _addr(y), x.size) and _host_flags(a) == [0, 0]
        z = d.gat_inverse(y, model)
        a = fake.last("b4d_gat_inverse_f32")
        _same_kind(z, xi, x.shape, "float32")
        assert (a["in"], a["out"], a["n"]) == (_addr(y), _addr(z), x.size) and _host_flags(a) == [0, 0]
        for quant, fn, dt in ((None, "b4d_denoise_vst_u16", "float32"),
                              ((1.0, 0.0, 2.0), "b4d_denoise_vst_q16_u16", "uint16")):
            y = d.denoise_vst(xi, model, 1.5, quantize=quant)
            a = fake.last(fn)
            _same_kind(y, xi, x.shape, dt)
            assert (a["in"], a["out"], a["n"], list(a["shape"]), a["sigma_vst"]) == (
                _addr(xi), _addr(y), 2, [6, 7, 8], 1.5)
            assert _host_flags(a) == [0, 0]


def test_coherence_and_small_calls(fake):
    import b4d

    d = _denoiser(fake)
    labels = np.ones(VOL.shape, np.uint64)
    raw = VOL.astype(np.float32)
    rej, tables = d.coherence_scores(labels, raw)
    a = fake.last("b4d_coherence_gate")
    assert rej.dtype == bool and rej.shape == (1,) and tables == [{}]
    assert (a["raw"], a["labels"], a["n"], a["lag"], a["in_on_device"]) == (raw.ctypes.data, labels.ctypes.data, 1, 2,
                                                                            0)
    assert d.patch_has_incoherent_segment(labels, raw) is False

    numq, wmap = d.debug_accumulators(10)
    a = fake.last("b4d_debug_accumulators")
    assert (a["numq"], a["wmap"], a["n"]) == (numq.ctypes.data, wmap.ctypes.data, 10) and numq.dtype == np.int64
    nu = np.ones(64, np.float32)
    d.set_noise_model(nu, nu)
    assert fake.last("b4d_set_noise_model")["nu_ht"] is not None
    d.set_noise_model()
    assert fake.last("b4d_set_noise_model")["nu_wie"] is None
    d.set_profile(b4d.BM4DProfile(max_stack_size_ht=8), stages=1)
    assert fake.calls[-1][0] == "b4d_set_profile"
    d.set_pass_voxels(1 << 33)
    assert fake.last("b4d_set_pass_voxels")["voxels"] == 1 << 33
    d.set_pipeline_min_voxels(7)
    assert fake.last("b4d_set_pipeline_min_voxels")["voxels"] == 7
    assert d.stream_ptr() == 0
    assert set(d.last_timings()) == set(b4d._lib.T_NAMES)
    assert set(d.last_match_stats()) == {"retry_refs", "wide_tiles", "slow_refs", "byte_tiles"}
    assert set(d.measure_pipe_peaks()) == {"imad", "iadd3", "sub_mad", "ffma"}


def test_wrong_dtype_or_ndim_never_reaches_the_library(fake):
    import b4d

    d = _denoiser(fake)
    model = b4d.PoissonGaussian(2.0, 10.0, 1.0)
    f32, i16, u16_2d = VOL.astype(np.float32), VOL.astype(np.int16), VOL[0]
    d.slab_stage1(VOL, 0, 6, 24.0)
    fake.calls.clear()
    bad = [
        lambda: d.denoise(i16, 24.0), lambda: d.denoise(u16_2d, 24.0), lambda: d.targets(VOL, 0.0, 24.0),
        lambda: d.targets(f32[None], 0.0, 24.0), lambda: d.denoise_slab(f32, 0, 6, 0, 6, 24.0),
        lambda: d.denoise_slab(VOL[None], 0, 6, 0, 6, 24.0), lambda: d.slab_stage1(i16, 0, 6, 24.0),
        lambda: d.slab_stage1(u16_2d, 0, 6, 24.0), lambda: d.denoise_quantized(f32, 24.0),
        lambda: d.match_stage1(f32, 24.0), lambda: d.match_stage1(u16_2d, 24.0),
        lambda: d.foreground_mask(f32), lambda: d.foreground_mask(u16_2d), lambda: d.chunk_shuffle(f32),
        lambda: d.chunk_shuffle(VOL[None]), lambda: d.tile_stats(f32), lambda: d.noise_sigma(f32),
        lambda: d.noise_sigma(u16_2d), lambda: d.noise_level_function(i16), lambda: d.noise_level_function(u16_2d),
        lambda: d.gat_forward(f32, model), lambda: d.gat_inverse(VOL, model), lambda: d.denoise_vst(f32, model),
        lambda: d.denoise_vst(u16_2d, model),
    ]
    for call in bad:
        with pytest.raises(ValueError):
            call()
    import torch

    for call in (lambda: d.denoise(torch.zeros((6, 7, 8), dtype=torch.int16), 24.0),
                 lambda: d.quantize(torch.zeros(5, dtype=torch.float64)),
                 lambda: d.slab_set_basic(0, torch.zeros((1, 7, 8), dtype=torch.float64)),
                 lambda: d.chunk_shuffle(torch.zeros((6, 7), dtype=torch.uint16))):
        with pytest.raises(ValueError):
            call()
    assert fake.calls == []


# ------------------------------------------------------- foreign device ----
@pytest.mark.gpu
def test_foreign_device_never_reaches_the_library():
    """A handle bound to cuda:0 refuses cuda:1 tensors and device="cuda:1" outputs with ValueError; the fake library
    behind it records that no call was made."""
    import torch

    import b4d

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    fake = FakeLib()
    d = _denoiser(fake, device=0)
    d._slab_shape = (6, 7, 8)
    model = b4d.PoissonGaussian(2.0, 10.0, 1.0)
    u = torch.from_numpy(VOL).to("cuda:1")
    f = u.float()
    calls = [
        lambda: d.denoise(u, 24.0), lambda: d.denoise(f, 24.0), lambda: d.denoise_slab(u, 0, 6, 0, 6, 24.0),
        lambda: d.denoise_slab(u, 0, 6, 0, 6, 24.0, quantize=(0.0, 0.0, 1.0)), lambda: d.slab_stage1(u, 0, 6, 24.0),
        lambda: d.slab_set_basic(0, f[:2]), lambda: d.denoise_quantized(u, 24.0), lambda: d.quantize(f),
        lambda: d.chunk_shuffle(u), lambda: d.tile_stats(u), lambda: d.noise_sigma(u),
        lambda: d.noise_level_function(u), lambda: d.gat_forward(u, model), lambda: d.gat_inverse(f, model),
        lambda: d.denoise_vst(u, model), lambda: d.denoise_vst(u, model, quantize=(0.0, 0.0, 1.0)),
        lambda: d.slab_basic(0, 2, device="cuda:1"), lambda: d.slab_stage2(0, 6, device="cuda:1"),
        lambda: d.slab_stage2(0, 6, device=torch.device("cuda", 1), quantize=(0.0, 0.0, 1.0)),
    ]
    for call in calls:
        with pytest.raises(ValueError):
            call()
    assert fake.calls == []
