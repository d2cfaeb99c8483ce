"""Host-side mirror of the reference's BM4D call surface, over libb4d.so.

What it replaces (paths under /root/reference/src/aind_exaspim_image_compression):

* ``bm4d(z, sigma_psd)``                     machine_learning/data_handling.py:332, :926;
                                             evaluate.py:202 (uint16, non-contiguous view)
* ``read_counts`` + ``bm4d`` + ``np.clip``   machine_learning/data_handling.py:315-354
                                             -> :func:`precompute_targets` (batched)
* clip + rint + uint16                       machine_learning/transforms.py:150-152, :403-411
                                             -> :func:`quantize`
* ``estimate_offset`` / median-MAD sigma     machine_learning/transforms.py:414-438,
                                             machine_learning/metrics.py:54-58 -> :func:`tile_stats`

Same names, argument meaning and error behaviour as the ``bm4d`` package's entry
point (``ValueError`` for shape/dtype, ``RuntimeError`` for CUDA,
``NotImplementedError`` for options outside the path).  NumPy in -> NumPy out; torch in ->
torch out on the same device.  Everything computes on the GPU through the C ABI;
there is no CPU fallback.
"""
import collections
import ctypes
import enum
import math
import os

import numpy as np

from . import _lib


class BM4DStages(enum.Enum):
    """Same members as ``bm4d.BM4DStages``."""

    HARD_THRESHOLDING = 1
    WIENER_FILTERING = 2
    ALL_STAGES = 3


class BM4DProfile:
    """Algorithm constants (SURVEY.md Appendix A).  Field names follow the
    ``bm4d`` package's profile where one exists; each maps onto ``b4d_profile``."""

    def __init__(self, **kw):
        self.bs_ht = (4, 4, 4)
        self.step_ht = (3, 3, 3)
        self.max_stack_size_ht = 16
        self.search_window_ht = (5, 5, 5)  # half-width per axis: window side 11
        self.tau_match_ht = 2.9527
        self.lambda_thr = 2.7
        self.bs_wiener = (4, 4, 4)
        self.step_wiener = (3, 3, 3)
        self.max_stack_size_wiener = 32
        self.search_window_wiener = (5, 5, 5)
        self.tau_match_wiener = 0.7693
        self.beta = 2.0  # Kaiser window parameter of the aggregation window
        self.deterministic = True  # always: fixed-point, order-independent aggregation (kept for compatibility)
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError("unknown profile field %r" % k)
            setattr(self, k, v)

    def key(self):
        return tuple(sorted((k, tuple(v) if np.ndim(v) else v) for k, v in vars(self).items()))

    def to_c(self, stages=2):
        def cube(v, name):
            v = tuple(int(x) for x in (v if np.ndim(v) else (v, v, v)))
            if len(set(v)) != 1:
                raise NotImplementedError("%s must be isotropic, got %r" % (name, v))
            return v[0]

        if cube(self.bs_ht, "bs_ht") != 4 or cube(self.bs_wiener, "bs_wiener") != 4:
            raise NotImplementedError("only 4x4x4 blocks are implemented")
        if cube(self.step_ht, "step_ht") != 3 or cube(self.step_wiener, "step_wiener") != 3:
            raise NotImplementedError("only step 3 is implemented")
        return _lib.default_profile(
            search_ht=2 * cube(self.search_window_ht, "search_window_ht") + 1,
            search_wie=2 * cube(self.search_window_wiener, "search_window_wiener") + 1,
            k_ht=int(self.max_stack_size_ht),
            k_wie=int(self.max_stack_size_wiener),
            tau_ht=float(self.tau_match_ht),
            tau_wie=float(self.tau_match_wiener),
            lambda_ht=float(self.lambda_thr),
            kaiser_beta=float(self.beta),
            deterministic=1 if self.deterministic else 0,
            stages=int(stages),
        )


def _profile_from_arg(profile):
    if isinstance(profile, BM4DProfile):
        return profile
    if profile is None or profile == "np":
        return BM4DProfile()
    raise ValueError("profile must be 'np' or a BM4DProfile, got %r" % (profile,))


def _is_torch(x):
    return type(x).__module__.split(".")[0] == "torch"


def _dtype_name(x):
    return str(x.dtype).replace("torch.", "")


def _array_arg(x, dtypes, ndims, what, cast=False):
    """Check an array argument before any handle or device work: a torch tensor, or anything np.asarray takes, of one
    of the dtype names `dtypes` and, unless `ndims` is None, of one of the dimensionalities `ndims`; ValueError
    otherwise.  With `cast`, NumPy input is first converted to dtypes[0] (a tensor must have it already).  Returns the
    tensor or the ndarray."""
    if not _is_torch(x):
        x = np.asarray(x, dtype=dtypes[0] if cast else None)
    dtype = _dtype_name(x)
    if dtype not in dtypes:
        raise ValueError("%s expects %s, got %s" % (what, " or ".join(dtypes), dtype))
    if ndims is not None and x.ndim not in ndims:
        raise ValueError("%s expects %s-D input, got %d-D" % (what, " or ".join(str(n) for n in ndims), x.ndim))
    return x


def _ptr(a):
    """Address of an array's data for a pointer parameter of the C ABI; None stays None (NULL)."""
    if a is None:
        return None
    return a.data_ptr() if _is_torch(a) else a.ctypes.data


def _out_like(x, shape, dtype):
    """New output of `shape` and dtype name `dtype` where the input x lives: torch on x's device, else NumPy."""
    if _is_torch(x):
        import torch

        return torch.empty(shape, dtype=getattr(torch, dtype), device=x.device)
    return np.empty(shape, dtype=dtype)


def _host_out(out, shape, dtype):
    """A caller's NumPy output (e.g. a pinned buffer), which must be C-contiguous of `shape` and `dtype`; a new array
    when `out` is None."""
    if out is None:
        return np.empty(shape, dtype=dtype)
    if out.shape != tuple(shape) or out.dtype != dtype or not out.flags.c_contiguous:
        raise ValueError("out must be a C-contiguous %s array of shape %r" % (np.dtype(dtype).name, tuple(shape)))
    return out


def _quantize_args(quantize):
    """quantize = (offset_sub, offset_add, step[, truncate]) -> the four trailing arguments of the *_q16 calls."""
    q = tuple(quantize) + (False,) * (4 - len(quantize))
    return q[0], q[1], q[2], int(bool(q[3]))


class StepTable(collections.namedtuple("StepTable", "steps tile")):
    """Per-tile quantizer steps (DESIGN §3 item 13): steps[ntz][nty][ntx] (float32) on the C-order grid of tiles of
    sides tile = (tz, ty, tx), anchored at the volume's plane 0 and ragged at the far faces -- the grid of noise_sigma's
    tiles and of the codec's chunks.  The voxel at global (z, y, x) is quantized with steps[z // tz][y // ty][x // tx],
    bit for bit as the scalar quantizer with that step.  A torch tensor is copied to the host."""

    __slots__ = ()

    def __new__(cls, steps, tile):
        if _is_torch(steps):
            steps = steps.detach().cpu().numpy()
        return super().__new__(cls, np.ascontiguousarray(steps, dtype=np.float32), tuple(int(t) for t in tile))


def _step_table_args(table, shape, z_begin=0, z_total=None):
    """Checks of a StepTable against the (D, H, W) planes of a call that start at global plane z_begin, before any
    handle work (ValueError).  z_total given (slab forms): the grid covers exactly z_total planes; else it must reach
    plane z_begin + D - 1.  Returns (steps, tile, grid) as the C ABI takes them."""
    steps, tile = table.steps, table.tile
    if steps.ndim != 3:
        raise ValueError("a step table must be 3-D (ntz, nty, ntx), got %d-D" % steps.ndim)
    if len(tile) != 3 or any(t < 1 for t in tile):
        raise ValueError("tile must be three sides >= 1, got %r" % (tile,))
    if not (np.all(np.isfinite(steps)) and np.all(steps >= 1)):
        raise ValueError("every step must be finite and >= 1")
    D, H, W = (int(v) for v in shape)
    ntz, nty, ntx = steps.shape
    if (nty, ntx) != (-(-H // tile[1]), -(-W // tile[2])):
        raise ValueError("step table grid (nty, ntx) = %r does not cover (H, W) = %r in tiles of %r"
                         % ((nty, ntx), (H, W), tile[1:]))
    if int(z_begin) < 0:
        raise ValueError("z_begin must be >= 0, got %r" % (z_begin,))
    if z_total is not None and ntz != -(-int(z_total) // tile[0]):
        raise ValueError("step table has %d tile layers; %d planes in tiles of %d need %d"
                         % (ntz, z_total, tile[0], -(-int(z_total) // tile[0])))
    if ntz * tile[0] < int(z_begin) + D:
        raise ValueError("planes [%d, %d) reach beyond the step table's %d tile layers of %d"
                         % (z_begin, int(z_begin) + D, ntz, tile[0]))
    return steps, _lib.shape3(tile), _lib.shape3(steps.shape)


def _table_of(quantize):
    """The StepTable of a quantize tuple, or None for a scalar step (or no quantize)."""
    if quantize is not None and len(quantize) >= 3 and isinstance(quantize[2], StepTable):
        return quantize[2]
    return None


class Denoiser:
    """One ``b4d_handle``: scratch buffers + a stream on one CUDA device.
    Not thread-safe; one per (process, device)."""

    def __init__(self, device=0, profile=None, stages=2):
        self.lib = _lib.load()
        self.device = int(device)
        self.profile = _profile_from_arg(profile)
        self._stages = stages
        self._h = ctypes.c_void_p()
        cprof = self.profile.to_c(stages)
        _lib.check(self.lib.b4d_create(self.device, ctypes.byref(cprof), ctypes.byref(self._h)))
        self._pid = os.getpid()

    def close(self):
        if getattr(self, "_h", None) and self._h and self._pid == os.getpid():
            self.lib.b4d_destroy(self._h)
        self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check_device(self, device):
        """ValueError unless the torch device `device` is this handle's CUDA device: the library would otherwise be
        handed a pointer into another GPU's memory."""
        if device.type != "cuda" or device.index != self.device:
            raise ValueError("%s is not the handle's device cuda:%d" % (device, self.device))

    def _input(self, x):
        """(keep-alive, pointer, on-device flag, shape) of an array that passed _array_arg.  A CUDA tensor must live on
        the handle's device; a tensor is made contiguous, and the current torch stream of its device is synchronised so
        that the library reads finished data.  NumPy input is made C-contiguous."""
        if not _is_torch(x):
            xc = np.ascontiguousarray(x)
            return xc, xc.ctypes.data, False, xc.shape
        if x.is_cuda:
            self._check_device(x.device)
        xc = x.contiguous()
        if xc.is_cuda:
            import torch

            torch.cuda.current_stream(xc.device).synchronize()
        return xc, xc.data_ptr(), xc.is_cuda, tuple(xc.shape)

    def _device_out(self, shape, dtype, device):
        """New torch output of dtype name `dtype` on `device`, which must be the handle's CUDA device ("cuda" without
        an index is the current device, as torch reads it)."""
        import torch

        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self._check_device(device)
        return torch.empty(shape, dtype=getattr(torch, dtype), device=device)

    def debug_accumulators(self, n):
        """(numq, wmap) int64 arrays: the fixed-point aggregation state the last filter stage of the last
        single-volume call left on the device (b4d_debug_accumulators; diagnostics for the parity tests)."""
        numq = np.empty(n, dtype=np.int64)
        wmap = np.empty(n, dtype=np.int64)
        _lib.check(self.lib.b4d_debug_accumulators(self._h, numq.ctypes.data, wmap.ctypes.data, n))
        return numq, wmap

    def set_noise_model(self, nu_ht=None, nu_wie=None):
        """Coloured noise: relative coefficient variances of the two block transforms (b4d_set_noise_model,
        see noise_model_from_psd); None, None switches back to white noise."""
        if nu_ht is None and nu_wie is None:
            _lib.check(self.lib.b4d_set_noise_model(self._h, None, None))
            return
        a = np.ascontiguousarray(nu_ht, dtype=np.float32).reshape(-1)
        b = np.ascontiguousarray(nu_wie, dtype=np.float32).reshape(-1)
        if a.size != 64 or b.size != 64:
            raise ValueError("nu_ht and nu_wie must hold 64 values each")
        _lib.check(self.lib.b4d_set_noise_model(self._h, a.ctypes.data, b.ctypes.data))

    def set_profile(self, profile=None, stages=2):
        """Switch algorithm constants (no-op when nothing changes)."""
        prof = _profile_from_arg(profile)
        if prof.key() == self.profile.key() and stages == self._stages:
            return
        cprof = prof.to_c(stages)
        _lib.check(self.lib.b4d_set_profile(self._h, ctypes.byref(cprof)))
        self.profile = prof
        self._stages = stages

    # ---- raw pointer level -------------------------------------------------
    def denoise_ptr(self, in_ptr, dtype, n, shape, sigma, out_ptr, in_dev, out_dev):
        fn = self.lib.b4d_denoise_u16 if dtype == np.uint16 else self.lib.b4d_denoise_f32
        _lib.check(fn(self._h, in_ptr, n, _lib.shape3(shape), sigma, out_ptr, int(in_dev), int(out_dev)))

    # ---- array level ---------------------------------------------------------
    def denoise(self, z, sigma):
        """(D,H,W) or (N,D,H,W); uint16 or float32; NumPy or torch -> float32."""
        zc, ptr, on_dev, shape = self._input(_array_arg(z, ("uint16", "float32"), (3, 4), "denoise"))
        out = _out_like(zc, shape, "float32")
        n = shape[0] if len(shape) == 4 else 1
        self.denoise_ptr(ptr, np.dtype(_dtype_name(zc)), n, shape[-3:], sigma, _ptr(out), on_dev, on_dev)
        return out

    def targets(self, raw_u16, offsets, sigma, max_count=65535.0, raw_out=None, teacher_out=None):
        """(N,D,H,W) uint16 patches + per-patch offsets -> (raw, teacher) float32 in one call
        (b4d_targets_u16: subtraction, BM4D and clip all on the device).  `raw_out` / `teacher_out`
        may be preallocated C-contiguous float32 arrays (e.g. the cache's memmaps)."""
        zc = np.ascontiguousarray(_array_arg(raw_u16, ("uint16",), (4,), "targets"))
        off = np.ascontiguousarray(np.broadcast_to(np.asarray(offsets, dtype=np.float32), (zc.shape[0],)))
        raw_out = _host_out(raw_out, zc.shape, np.float32)
        teacher_out = _host_out(teacher_out, zc.shape, np.float32)
        _lib.check(self.lib.b4d_targets_u16(self._h, zc.ctypes.data, zc.shape[0], _lib.shape3(zc.shape[1:]),
                                            off.ctypes.data, sigma, max_count, raw_out.ctypes.data,
                                            teacher_out.ctypes.data, 0, 0))
        return raw_out, teacher_out

    def denoise_slab(self, slab, z_begin, z_total, own_begin, own_end, sigma, out=None, quantize=None):
        """One z-slab (uint16, with halos) of a larger volume -> float32 owned planes.
        `out` (NumPy path only) receives the result in place, e.g. a pinned buffer.
        quantize = (offset_sub, offset_add, step[, truncate]): the fused denoise -> offset -> quantize path, the
        result is the uint16 volume K7 would give on the float32 output (2 bytes per voxel leave the device).  step
        may be a StepTable of the whole z_total-plane volume."""
        slab = _array_arg(slab, ("uint16",), (3,), "denoise_slab")
        table = _table_of(quantize)
        targs = _step_table_args(table, slab.shape, z_begin, z_total) if table is not None else None
        sc, in_ptr, on_dev, shape = self._input(slab)
        odt = "float32" if quantize is None else "uint16"
        oshape = (own_end - own_begin,) + shape[1:]
        out = _out_like(sc, oshape, odt) if _is_torch(sc) else _host_out(out, oshape, odt)
        if targs is not None:
            sub, add, _, trunc = _quantize_args(quantize)
            steps, tile, grid = targs
            _lib.check(self.lib.b4d_denoise_slab_qt16_u16(self._h, in_ptr, _lib.shape3(shape), z_begin, z_total,
                                                          own_begin, own_end, sigma, sub, add, tile, grid,
                                                          steps.ctypes.data, trunc, _ptr(out), on_dev, on_dev))
        elif quantize is None:
            _lib.check(self.lib.b4d_denoise_slab_u16(self._h, in_ptr, _lib.shape3(shape), z_begin, z_total, own_begin,
                                                     own_end, sigma, _ptr(out), on_dev, on_dev))
        else:
            _lib.check(self.lib.b4d_denoise_slab_q16_u16(self._h, in_ptr, _lib.shape3(shape), z_begin, z_total,
                                                         own_begin, own_end, sigma, *_quantize_args(quantize),
                                                         _ptr(out), on_dev, on_dev))
        return out

    # ---- the slab in two calls, for one neighbour exchange between the stages ----
    def slab_stage1(self, slab, z_begin, z_total, sigma):
        """Stage 1 on a uint16 slab (NumPy or torch); the basic estimate stays on the device."""
        sc, ptr, on_dev, shape = self._input(_array_arg(slab, ("uint16",), (3,), "slab_stage1"))
        self._slab_shape = tuple(int(v) for v in shape)
        self._slab_z = (int(z_begin), int(z_total), False)
        _lib.check(self.lib.b4d_slab_stage1_u16(self._h, ptr, _lib.shape3(shape), z_begin, z_total, sigma, on_dev))

    def slab_basic(self, plane0, nplanes, device=None):
        """Planes [plane0, plane0 + nplanes) (slab-local) of the basic estimate: a torch CUDA
        tensor when `device` is given, else a NumPy array."""
        shape = (int(nplanes),) + self._slab_shape[1:]
        buf = np.empty(shape, dtype=np.float32) if device is None else self._device_out(shape, "float32", device)
        if nplanes:
            _lib.check(self.lib.b4d_slab_basic_planes(self._h, plane0, nplanes, _ptr(buf), 0, device is not None))
        return buf

    def slab_set_basic(self, plane0, planes):
        """Overwrite planes of the basic estimate (the neighbour's exact halo planes)."""
        pc, ptr, on_dev, shape = self._input(_array_arg(planes, ("float32",), None, "slab_set_basic", cast=True))
        if tuple(shape[1:]) != self._slab_shape[1:]:
            raise ValueError("planes must have the slab's (H, W)")
        if shape[0]:
            _lib.check(self.lib.b4d_slab_basic_planes(self._h, plane0, shape[0], ptr, 1, on_dev))

    def slab_basic_tensor(self, device):
        """Zero-copy torch view (D, H, W) float32 of the open slab's basic estimate on `device`: a neighbour
        exchange reads the owned planes and writes the halo planes in place (b4d_slab_basic_ptr)."""
        import torch

        ptr = self.lib.b4d_slab_basic_ptr(self._h)
        if not ptr:
            _lib.check(-1)
        shape = tuple(int(v) for v in self._slab_shape)

        class _View:  # the CUDA array interface torch.as_tensor understands
            __cuda_array_interface__ = {"shape": shape, "typestr": "<f4", "data": (int(ptr), False), "version": 3,
                                        "strides": None}

        return torch.as_tensor(_View(), device=device)

    def slab_stage2_begin(self, own_begin, own_end):
        """Launch, without waiting, the part of the stage-2 front end that reads owned planes only."""
        _lib.check(self.lib.b4d_slab_stage2_begin(self._h, own_begin, own_end))

    def slab_stage2(self, own_begin, own_end, out=None, device=None, quantize=None):
        """Stage 2 on the completed basic estimate -> float32 owned planes (NumPy, or torch on
        `device`; `out` may be a preallocated NumPy array, e.g. pinned).  quantize = (offset_sub, offset_add,
        step[, truncate]): uint16 output of the fused quantizer instead (see denoise_slab); step may be a StepTable
        of the whole volume (not after slab_stage1_vst)."""
        table = _table_of(quantize)
        if table is not None:
            if getattr(self, "_slab_z", None) is None:
                raise ValueError("slab_stage1 has not been called")
            z_begin, z_total, vst = self._slab_z
            if vst:
                raise NotImplementedError("a step table on the VST path is not implemented")
            steps, tile, grid = _step_table_args(table, self._slab_shape, z_begin, z_total)
        oshape = (int(own_end - own_begin),) + self._slab_shape[1:]
        odt = "float32" if quantize is None else "uint16"
        out = _host_out(out, oshape, odt) if device is None else self._device_out(oshape, odt, device)
        on_dev = device is not None
        if table is not None:
            sub, add, _, trunc = _quantize_args(quantize)
            _lib.check(self.lib.b4d_slab_stage2_qt16(self._h, own_begin, own_end, sub, add, tile, grid,
                                                     steps.ctypes.data, trunc, _ptr(out), on_dev))
        elif quantize is None:
            _lib.check(self.lib.b4d_slab_stage2(self._h, own_begin, own_end, _ptr(out), on_dev))
        else:
            _lib.check(self.lib.b4d_slab_stage2_q16(self._h, own_begin, own_end, *_quantize_args(quantize), _ptr(out),
                                                    on_dev))
        return out

    def denoise_quantized(self, vol, sigma, offset_sub=0.0, offset_add=0.0, step=1.0, truncate=False, out=None):
        """denoise -> offset -> quantize of one uint16 volume in one call (b4d_denoise_q16_u16): the uint16 volume
        `quantize(denoise(vol, sigma), offset_sub, offset_add, step, truncate)` would give, bit for bit.  step may be
        a StepTable (b4d_denoise_slab_qt16_u16 on the slab 0, D, 0, D)."""
        D = int(vol.shape[0])
        return self.denoise_slab(vol, 0, D, 0, D, sigma, out=out, quantize=(offset_sub, offset_add, step, truncate))

    def match_stage1(self, vol, sigma):
        """Instrumented stage-1 matcher: (idx[R,K] int32, ssd[R,K] uint64, count[R] int32)."""
        vol = np.ascontiguousarray(_array_arg(vol, ("uint16",), (3,), "match_stage1"))
        shape = _lib.shape3(vol.shape)
        R = self.lib.b4d_num_refs(shape)
        K = int(self.profile.max_stack_size_ht)
        idx = np.empty((R, K), dtype=np.int32)
        ssd = np.empty((R, K), dtype=np.uint64)
        cnt = np.empty((R,), dtype=np.int32)
        _lib.check(self.lib.b4d_match_stage1(self._h, vol.ctypes.data, shape, sigma, idx.ctypes.data, ssd.ctypes.data,
                                             cnt.ctypes.data))
        return idx, ssd, cnt

    def quantize(self, x, offset_sub=0.0, offset_add=0.0, step=1.0, truncate=False, z_begin=0):
        """K7: rint(clip((x - offset_sub + offset_add)/step, 0, 65535/step)) -> uint16.
        truncate=True: the evaluator's variant, np.maximum(v, 0).astype(int) cast to uint16 (evaluate.py:202,
        utils/img_util.py:420-423): toward zero, no upper clip, wrapping modulo 2^16.
        step may be a StepTable: x is then 3-D, planes [z_begin, z_begin + D) of the volume the table covers, and
        every voxel takes the step of its tile (b4d_quantize_tiled_u16)."""
        if isinstance(step, StepTable):
            x = _array_arg(x, ("float32",), (3,), "quantize", cast=True)
            steps, tile, grid = _step_table_args(step, x.shape, z_begin)
            xc, in_ptr, on_dev, shape = self._input(x)
            out = _out_like(xc, shape, "uint16")
            _lib.check(self.lib.b4d_quantize_tiled_u16(self._h, in_ptr, _lib.shape3(shape), int(z_begin), tile, grid,
                                                       steps.ctypes.data, offset_sub, offset_add, int(bool(truncate)),
                                                       _ptr(out), on_dev, on_dev))
            return out
        xc, in_ptr, on_dev, shape = self._input(_array_arg(x, ("float32",), None, "quantize", cast=True))
        out = _out_like(xc, shape, "uint16")
        fn = self.lib.b4d_quantize_trunc_u16 if truncate else self.lib.b4d_quantize_u16
        _lib.check(fn(self._h, in_ptr, math.prod(shape), offset_sub, offset_add, step, _ptr(out), on_dev, on_dev))
        return out

    def dequantize(self, q, step, offset_sub=0.0, offset_add=0.0, z_begin=0):
        """Inverse of quantize: x = ((float)q * s) + offset_sub - offset_add per voxel, each operation one float32
        IEEE operation (b4d_dequantize_tiled_f32).  q: 3-D uint16, planes [z_begin, z_begin + D) of the volume; step:
        a scalar (one tile) or a StepTable.  Within the clip range of the rounding quantizer |x - original| <= s / 2
        up to float32 rounding; the truncating quantizer's values come back biased low."""
        q = _array_arg(q, ("uint16",), (3,), "dequantize")
        if not isinstance(step, StepTable):
            step = StepTable(np.full((1, 1, 1), step, np.float32), (int(z_begin) + int(q.shape[0]),) + tuple(q.shape[1:]))
        steps, tile, grid = _step_table_args(step, q.shape, z_begin)
        qc, in_ptr, on_dev, shape = self._input(q)
        out = _out_like(qc, shape, "float32")
        _lib.check(self.lib.b4d_dequantize_tiled_f32(self._h, in_ptr, _lib.shape3(shape), int(z_begin), tile, grid,
                                                     steps.ctypes.data, offset_sub, offset_add, _ptr(out), on_dev,
                                                     on_dev))
        return out

    def set_pass_voxels(self, voxels):
        """Voxels per pass (scratch ~45 B each; 0 = default 1.25 Gi).  A uint16 volume larger than a
        pass is denoised as consecutive z-slabs with halos, by denoise and by denoise_vst (which first
        takes the value set of the whole volume); the result does not change."""
        _lib.check(self.lib.b4d_set_pass_voxels(self._h, int(voxels)))

    def set_pipeline_min_voxels(self, voxels):
        """Volume size from which host transfers are pipelined against the kernels (default 2^26)."""
        _lib.check(self.lib.b4d_set_pipeline_min_voxels(self._h, int(voxels)))

    def foreground_mask(self, raw_u16, offsets=0.0, k=6.0, dilate=1):
        """make_foreground_mask (metrics.py:32-61) of uint16 patches after the offset subtraction
        (data_handling.py:353-354): (D,H,W) or (N,D,H,W) uint16 -> bool mask of the same shape."""
        zc = np.ascontiguousarray(_array_arg(raw_u16, ("uint16",), (3, 4), "foreground_mask"))
        n = zc.shape[0] if zc.ndim == 4 else 1
        off = np.ascontiguousarray(np.broadcast_to(np.asarray(offsets, dtype=np.float32), (n,)))
        out = np.empty(zc.shape, dtype=np.uint8)
        _lib.check(self.lib.b4d_foreground_mask_u16(self._h, zc.ctypes.data, n, _lib.shape3(zc.shape[-3:]),
                                                    off.ctypes.data, k, int(dilate), out.ctypes.data, 0, 0))
        return out.view(np.bool_)

    def chunk_shuffle(self, x, chunk=(64, 64, 64), want_bytes=True, want_hist=True):
        """K9: C-order chunk gather + Blosc 2-byte shuffle of a uint16 volume, plus per-piece byte
        histograms [pieces, 2, 256] (uint32; int32 for torch input).  Returns (bytes or None, hist or None)."""
        if len(chunk) != 3:
            raise ValueError("chunk must have three entries")
        if not (want_bytes or want_hist):
            raise ValueError("nothing requested")
        xc, in_ptr, on_dev, shape = self._input(_array_arg(x, ("uint16",), (3,), "chunk_shuffle"))
        npieces = 1
        for s_, c_ in zip(shape, chunk):
            if int(c_) < 1:
                raise ValueError("chunk sides must be >= 1")
            npieces *= -(-int(s_) // int(c_))
        out = _out_like(xc, (2 * math.prod(shape),), "uint8") if want_bytes else None
        hist = _out_like(xc, (npieces, 2, 256), "int32" if _is_torch(xc) else "uint32") if want_hist else None
        _lib.check(self.lib.b4d_chunk_shuffle_u16(self._h, in_ptr, _lib.shape3(shape), _lib.shape3(chunk), _ptr(out),
                                                  _ptr(hist), on_dev, on_dev))
        return out, hist

    def tile_stats(self, x, percentile=1.0, return_hist=False):
        """K8: offset percentile over non-zero voxels + median / MAD sigma of a uint16 tile."""
        xc, in_ptr, on_dev, shape = self._input(_array_arg(x, ("uint16",), None, "tile_stats"))
        st = _lib.Stats()
        hist = np.empty(65536, dtype=np.int64) if return_hist else None
        _lib.check(self.lib.b4d_tile_stats(self._h, in_ptr, math.prod(shape), percentile, ctypes.byref(st), _ptr(hist),
                                           on_dev))
        d = {k: getattr(st, k) for k, _ in _lib.Stats._fields_}
        return (d, hist) if return_hist else d

    def noise_sigma(self, x, tile=None, return_hist=False):
        """Noise standard deviation per tile from the MAD of the finest 3-D Haar detail (DESIGN §3.11).

        x     (D,H,W) or (N,D,H,W) uint16, NumPy or torch (host or CUDA).
        tile  (tz, ty, tx), even sides: a C-order grid anchored at the origin, ragged at the far faces;
              None: one tile per volume.
        Returns {"sigma", "mad", "cells"} (float64, float64, int64) shaped (N,)? + tile grid (the grid axes are
        dropped when tile is None); with return_hist, also the exact 262141-bin histogram of |d| over every cell
        of the call (int64), the payload to sum across ranks for noise_sigma_from_hist."""
        x, tile, grid = _noise_sigma_args(x, tile)
        xc, in_ptr, on_dev, shape = self._input(x)
        n = 1 if len(shape) == 3 else shape[0]
        out_shape = (() if len(shape) == 3 else (n,)) + grid
        sigma = np.empty(out_shape, np.float64)
        mad = np.empty(out_shape, np.float64)
        cells = np.empty(out_shape, np.int64)
        hist = np.empty(_lib.NOISE_HIST_BINS, np.int64) if return_hist else None
        _lib.check(
            self.lib.b4d_noise_sigma_u16(
                self._h, in_ptr, n, _lib.shape3(shape[-3:]), _lib.shape3(tile) if tile is not None else None,
                sigma.ctypes.data, mad.ctypes.data, cells.ctypes.data, _ptr(hist), on_dev,
            )
        )
        d = {"sigma": sigma[()], "mad": mad[()], "cells": cells[()]}
        return (d, hist) if return_hist else d

    # ---- Poisson-Gaussian noise (DESIGN §3.12) -------------------------------
    def noise_level_function(self, x, edges=None, min_cells=256):
        """Noise-level function var(z) = a E[z] + b of Poisson-Gaussian counts (DESIGN §3.12): the Haar-detail MAD of
        noise_sigma per intensity bin of the 2x2x2 cells, and a weighted least-squares line through the bins.

        x          (D,H,W) or (N,D,H,W) uint16, NumPy or torch (host or CUDA); one set of bins for every volume.
        edges      nb + 1 strictly increasing finite bin edges in counts (1 <= nb <= 64); a cell whose 8 voxels sum to
                   s is in bin k iff 8 edges[k] <= s < 8 edges[k + 1].  None: default_nlf_edges().
        min_cells  bins with fewer cells stay out of the fit.
        Returns {"edges", "cells", "level_sum", "level", "mad", "sigma", "a", "b", "usable"}: per-bin int64 / float64
        arrays (level = mean intensity of the bin's cells, NaN when empty), the fitted a, b (NaN when fewer than 2
        bins are usable) and the number of usable bins."""
        x, edges, min_cells = _nlf_args(x, edges, min_cells)
        xc, in_ptr, on_dev, shape = self._input(x)
        nb = edges.size - 1
        cells = np.empty(nb, np.int64)
        level_sum = np.empty(nb, np.int64)
        mad = np.empty(nb, np.float64)
        sigma = np.empty(nb, np.float64)
        level = np.empty(nb, np.float64)
        fit = np.empty(2, np.float64)
        usable = np.empty(1, np.int64)
        n = 1 if len(shape) == 3 else shape[0]
        _lib.check(
            self.lib.b4d_noise_level_u16(
                self._h, in_ptr, n, _lib.shape3(shape[-3:]), edges.ctypes.data, nb, min_cells, cells.ctypes.data,
                level_sum.ctypes.data, mad.ctypes.data, sigma.ctypes.data, level.ctypes.data, fit.ctypes.data,
                usable.ctypes.data, on_dev,
            )
        )
        return {"edges": edges, "cells": cells, "level_sum": level_sum, "level": level, "mad": mad, "sigma": sigma,
                "a": fit[0], "b": fit[1], "usable": int(usable[0])}

    def gat_forward(self, x, model):
        """Generalized Anscombe transform of uint16 counts under `model` (PoissonGaussian) -> float32, elementwise:
        2 sqrt(max((z - offset)/gain + 3/8 + (read_sigma/gain)^2, 0)), float64 inside.  NumPy or torch (host or
        CUDA) -> the same kind, same shape."""
        x = _array_arg(x, ("uint16",), None, "gat_forward")
        m = _model_c(model)
        xc, in_ptr, on_dev, shape = self._input(x)
        out = _out_like(xc, shape, "float32")
        _lib.check(self.lib.b4d_gat_forward_u16(self._h, ctypes.byref(m), in_ptr, math.prod(shape), _ptr(out), on_dev,
                                                on_dev))
        return out

    def gat_inverse(self, y, model):
        """Closed-form approximation of the exact unbiased inverse of gat_forward (Makitalo & Foi 2013), float32 ->
        float32 counts gain * lambda + offset; lambda = 0 for y <= sqrt(1.5)."""
        y = _array_arg(y, ("float32",), None, "gat_inverse")
        m = _model_c(model)
        yc, in_ptr, on_dev, shape = self._input(y)
        out = _out_like(yc, shape, "float32")
        _lib.check(self.lib.b4d_gat_inverse_f32(self._h, ctypes.byref(m), in_ptr, math.prod(shape), _ptr(out), on_dev,
                                                on_dev))
        return out

    def denoise_vst(self, x, model, sigma=1.0, quantize=None):
        """Denoise Poisson-Gaussian uint16 counts: gat_inverse(denoise(gat_forward(x, model), sigma), model), with the
        intermediate float32 volume never leaving the device.  sigma is the noise level after the transform: 1 for an
        exact model.  (D,H,W) or (N,D,H,W), NumPy or torch -> float32; quantize = (offset_sub, offset_add, step[,
        truncate]): the uint16 volume quantize() gives on that float32 result instead.  A volume larger than a pass
        (set_pass_voxels) is denoised as z-slabs with the value set of the whole volume: the same result."""
        x = _vst_args(x, sigma, quantize)
        m = _model_c(model)
        xc, in_ptr, on_dev, shape = self._input(x)
        n = 1 if len(shape) == 3 else shape[0]
        out = _out_like(xc, shape, "float32" if quantize is None else "uint16")
        if quantize is None:
            _lib.check(self.lib.b4d_denoise_vst_u16(self._h, in_ptr, n, _lib.shape3(shape[-3:]), ctypes.byref(m), sigma,
                                                    _ptr(out), on_dev, on_dev))
        else:
            _lib.check(self.lib.b4d_denoise_vst_q16_u16(self._h, in_ptr, n, _lib.shape3(shape[-3:]), ctypes.byref(m),
                                                        sigma, *_quantize_args(quantize), _ptr(out), on_dev, on_dev))
        return out

    def denoise_slab_vst(self, slab, z_begin, z_total, own_begin, own_end, model, value_hist, first, sigma=1.0,
                         out=None, quantize=None):
        """denoise_slab through the GAT: one z-slab (uint16, with halos) of a larger volume -> its owned planes of
        denoise_vst on the whole volume, bit for bit (DESIGN §3.12, map rule).  value_hist: the 65536 counts of every
        uint16 value of the WHOLE volume (tile_stats(..., return_hist=True), or such histograms summed across ranks);
        first: the whole volume's voxel (0, 0, 0).  out / quantize as denoise_slab."""
        sc, in_ptr, on_dev, shape = self._input(_vst_args(slab, sigma, quantize, (3,), "denoise_slab_vst"))
        m, hist, first = _model_c(model), _value_hist(value_hist), int(first)
        odt = "float32" if quantize is None else "uint16"
        oshape = (own_end - own_begin,) + shape[1:]
        out = _out_like(sc, oshape, odt) if _is_torch(sc) else _host_out(out, oshape, odt)
        if quantize is None:
            _lib.check(self.lib.b4d_denoise_slab_vst_u16(self._h, in_ptr, _lib.shape3(shape), z_begin, z_total,
                                                         own_begin, own_end, ctypes.byref(m), sigma, hist.ctypes.data,
                                                         first, _ptr(out), on_dev, on_dev))
        else:
            _lib.check(self.lib.b4d_denoise_slab_vst_q16_u16(self._h, in_ptr, _lib.shape3(shape), z_begin, z_total,
                                                             own_begin, own_end, ctypes.byref(m), sigma,
                                                             hist.ctypes.data, first, *_quantize_args(quantize),
                                                             _ptr(out), on_dev, on_dev))
        return out

    def slab_stage1_vst(self, slab, z_begin, z_total, model, value_hist, first, sigma=1.0):
        """slab_stage1 through the GAT (value_hist, first as denoise_slab_vst); slab_basic / slab_set_basic /
        slab_basic_tensor / slab_stage2_begin / slab_stage2 complete it, and stage 2 ends in the inverse."""
        sc, ptr, on_dev, shape = self._input(_vst_args(slab, sigma, None, (3,), "slab_stage1_vst"))
        m, hist, first = _model_c(model), _value_hist(value_hist), int(first)
        self._slab_shape = tuple(int(v) for v in shape)
        self._slab_z = (int(z_begin), int(z_total), True)
        _lib.check(self.lib.b4d_slab_stage1_vst_u16(self._h, ptr, _lib.shape3(shape), z_begin, z_total,
                                                    ctypes.byref(m), sigma, hist.ctypes.data, first, on_dev))

    def coherence_scores(self, labels, raw, smooth_sigma=1.0, coherence_lag=2, min_autocorr=0.4,
                         max_highfreq_frac=0.35, min_segment_voxels=50, max_segments=1024):
        """The spatial-coherence gate of the sampler (metrics.py:189-260) on the device, for one patch (3-D arrays)
        or a batch (4-D): returns (reject[n] bool, [ {label: (voxels, autocorr, highfreq)} per patch ])."""
        lab = np.ascontiguousarray(labels, dtype=np.uint64)
        x = np.ascontiguousarray(raw, dtype=np.float32)
        if lab.shape != x.shape or x.ndim not in (3, 4):
            raise ValueError("labels and raw must be 3-D (or batched 4-D) arrays of the same shape")
        n = 1 if x.ndim == 3 else x.shape[0]
        shape = x.shape[-3:]
        reject = np.zeros(n, dtype=np.uint8)
        seg = (_lib.SegmentScore * (n * max_segments))()
        cnt = np.zeros(n, dtype=np.int64)
        _lib.check(
            self.lib.b4d_coherence_gate(
                self._h, x.ctypes.data, lab.ctypes.data, n, _lib.shape3(shape), min_autocorr, max_highfreq_frac,
                min_segment_voxels, smooth_sigma, coherence_lag, reject.ctypes.data, seg, max_segments,
                cnt.ctypes.data, 0,
            )
        )
        tables = []
        for i in range(n):
            if cnt[i] > max_segments:
                raise ValueError("patch %d holds %d segments, max_segments is %d" % (i, cnt[i], max_segments))
            tables.append({int(seg[i * max_segments + j].label): (int(seg[i * max_segments + j].voxels),
                                                                   float(seg[i * max_segments + j].autocorr),
                                                                   float(seg[i * max_segments + j].highfreq))
                           for j in range(int(cnt[i]))})
        return reject.astype(bool), tables

    def patch_has_incoherent_segment(self, labels, raw, min_autocorr=0.4, max_highfreq_frac=0.35,
                                     min_segment_voxels=50, smooth_sigma=1.0, coherence_lag=2):
        """Drop-in for metrics.patch_has_incoherent_segment (same arguments, same bool); a 4-D batch returns one bool
        per patch."""
        rej, _ = self.coherence_scores(labels, raw, smooth_sigma, coherence_lag, min_autocorr, max_highfreq_frac,
                                       min_segment_voxels)
        return bool(rej[0]) if np.ndim(raw) == 3 else rej

    def stream_ptr(self):
        """cudaStream_t of the handle (int): wrap it in torch.cuda.ExternalStream to
        record CUDA events around calls."""
        return int(self.lib.b4d_stream(self._h) or 0)

    def last_timings(self):
        ms = (ctypes.c_float * _lib.T_COUNT)()
        nl = (ctypes.c_int64 * _lib.T_COUNT)()
        _lib.check(self.lib.b4d_last_timings(self._h, ms, nl))
        return {name: (float(ms[i]), int(nl[i])) for i, name in enumerate(_lib.T_NAMES)}

    def last_match_stats(self):
        out = (ctypes.c_uint64 * 4)()
        _lib.check(self.lib.b4d_last_match_stats(self._h, out))
        return {"retry_refs": int(out[0]), "wide_tiles": int(out[1]), "slow_refs": int(out[2]), "byte_tiles": int(out[3])}

    def measure_pipe_peaks(self):
        out = (ctypes.c_double * 4)()
        _lib.check(self.lib.b4d_measure_pipe_peaks(self._h, out))
        return {"imad": out[0], "iadd3": out[1], "sub_mad": out[2], "ffma": out[3]}


# --------------------------------------------------------------------------
# module-level call surface (lazy per-process handles: the reference calls
# bm4d() from forked ProcessPool workers, scripts/precompute.py:215-222)
# --------------------------------------------------------------------------
_handles = {}


def get_denoiser(device=None):
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if "B4D_DEVICE" not in os.environ else int(
            os.environ["B4D_DEVICE"]
        )
    key = (os.getpid(), int(device))
    h = _handles.get(key)
    if h is None:
        h = Denoiser(device)
        _handles[key] = h
    return h


def _sigma_scalar(sigma_psd):
    s = np.asarray(sigma_psd, dtype=np.float64)
    if s.ndim == 0 or s.size == 1:
        return float(s.reshape(-1)[0])
    if np.all(s == s.reshape(-1)[0]):
        # a constant PSD of an N-voxel transform equals sigma^2 * N (white noise)
        return float(np.sqrt(s.reshape(-1)[0] / s.size))
    raise NotImplementedError("a coloured-noise PSD is accepted by bm4d() only; this entry point takes a scalar sigma")


_HAAR4 = np.array([[0.5, 0.5, 0.5, 0.5], [0.5, 0.5, -0.5, -0.5], [np.sqrt(0.5), -np.sqrt(0.5), 0.0, 0.0],
                   [0.0, 0.0, np.sqrt(0.5), -np.sqrt(0.5)]])
_DCT4 = np.array([[(0.5 if k == 0 else np.sqrt(0.5)) * np.cos(np.pi * (2 * n + 1) * k / 8.0) for n in range(4)]
                  for k in range(4)])


def noise_model_from_psd(psd):
    """Reduce a noise PSD to what the kernels need (include/b4d.h, b4d_set_noise_model): (sigma, nu_ht[64],
    nu_wie[64]) — the root of the mean noise variance and, for the stage-1 (Haar = bior1.5 at length 4) and stage-2
    (DCT-II) block transforms, the relative variance of each of the 64 coefficients of a 4^3 block of that noise.

    ``psd`` is the array form of bm4d's ``sigma_psd``: E|FFT(noise)|^2 on the grid of the volume (or any grid of at
    least 4 points per axis), unnormalised DFT, so that white noise of standard deviation s has psd == s^2 * psd.size.
    The autocovariance r = ifftn(psd) / psd.size gives the covariance C[u, v] = r[u - v] of the 64 voxels of a
    block; coefficient c of the orthonormal transform T has the variance (T C T^t)[c, c]."""
    P = np.asarray(psd, dtype=np.float64)
    if P.ndim != 3 or min(P.shape) < 4:
        raise ValueError("a noise PSD must be a 3-D array with at least 4 points per axis")
    if not np.all(np.isfinite(P)) or P.min() < 0 or P.max() <= 0:
        raise ValueError("a noise PSD must be finite, non-negative and not identically zero")
    r = np.real(np.fft.ifftn(P)) / P.size
    idx = np.arange(4)
    d = idx[:, None] - idx[None, :]  # u - v per axis
    C = r[np.ix_(*[np.arange(-3, 4) % n for n in P.shape])]  # offsets -3 .. 3 per axis, as a 7^3 cube
    cov = C[(d + 3)[:, None, None, :, None, None], (d + 3)[None, :, None, None, :, None],
            (d + 3)[None, None, :, None, None, :]].reshape(64, 64)
    sigma2 = float(r[0, 0, 0])
    out = []
    for t1 in (_HAAR4, _DCT4):
        T = np.kron(t1, np.kron(t1, t1))  # index (z*4 + y)*4 + x on both sides
        var = np.einsum("cu,uv,cv->c", T, cov, T)
        out.append(np.maximum(var / sigma2, 1e-12).astype(np.float32))
    return float(np.sqrt(sigma2)), out[0], out[1]


def _prepare(z):
    """dtype contract of the drop-in: returns (array for the C ABI, output cast)."""
    if _is_torch(z):
        return z, None
    z = np.asarray(z)
    if z.dtype == np.uint16 or z.dtype == np.float32:
        return z, None
    if z.dtype.kind in "iu" or z.dtype == np.bool_:
        if z.size and (z.min() < 0 or z.max() > 65535):
            return z.astype(np.float32), None
        return z.astype(np.uint16), None
    if z.dtype.kind == "f":
        return z.astype(np.float32), z.dtype
    raise ValueError("unsupported dtype %s" % z.dtype)


def bm4d(z, sigma_psd, profile="np", stage_arg=BM4DStages.ALL_STAGES, blockmatches=(False, False), device=None):
    """Drop-in for ``bm4d.bm4d``: denoise one 3-D volume.

    z          NumPy or torch, 3-D, uint16 or float32 (other real dtypes are
               converted), any strides.
    sigma_psd  noise standard deviation in the units of ``z`` (scalar), or the noise PSD as a 3-D array
               (E|FFT(noise)|^2, unnormalised DFT: white noise of std s is s^2 * size) for coloured noise.
    Returns a new array of the same shape: float32 (input dtype for float64).
    Unclipped — callers clip (data_handling.py:333, evaluate.py:202).
    """
    if blockmatches not in ((False, False), [False, False], None):
        raise NotImplementedError("returning / reusing block matches is not implemented")
    if isinstance(stage_arg, BM4DStages):
        if stage_arg == BM4DStages.WIENER_FILTERING:
            raise ValueError("WIENER_FILTERING alone needs a basic estimate; pass ALL_STAGES")
        stages = 1 if stage_arg == BM4DStages.HARD_THRESHOLDING else 2
    else:
        raise NotImplementedError("passing a basic estimate as stage_arg is not implemented")
    if np.ndim(z) != 3 if not _is_torch(z) else z.ndim != 3:
        raise ValueError("bm4d expects a 3-D array, got %d-D" % (z.ndim if _is_torch(z) else np.ndim(z)))
    h = get_denoiser(device)
    h.set_profile(profile, stages)
    zz, cast = _prepare(z)
    s = np.asarray(sigma_psd, dtype=np.float64)
    if s.ndim == 3 and s.size > 1 and not np.all(s == s.reshape(-1)[0]):
        # coloured noise: per-coefficient variances of both block transforms (a constant PSD is white noise and
        # takes the scalar path, bit for bit)
        sigma, nu_ht, nu_wie = noise_model_from_psd(s)
        h.set_noise_model(nu_ht, nu_wie)
        try:
            out = h.denoise(zz, sigma)
        finally:
            h.set_noise_model(None, None)
    else:
        out = h.denoise(zz, _sigma_scalar(sigma_psd))
    return out.astype(cast) if cast is not None else out


def bm4d_batch(patches, sigma, profile="np", device=None):
    """N independent equal-shape patches in one call: (N,D,H,W) -> float32."""
    h = get_denoiser(device)
    h.set_profile(profile, 2)
    zz, _ = _prepare(patches)
    if zz.ndim != 4:
        raise ValueError("bm4d_batch expects (N, D, H, W)")
    return h.denoise(zz, _sigma_scalar(sigma))


def precompute_targets(raw_u16, offsets, sigma, max_count=65535.0, device=None):
    """Batched ``_sample_counts`` core (data_handling.py:315-354):
    raw = uint16 -> float32 - offset; teacher = clip(bm4d(raw, sigma), 0, max_count).

    raw_u16  (N,D,H,W) uint16;  offsets scalar or (N,) per-patch scalars.
    Returns (raw float32, teacher float32) as the cache stores them
    (scripts/precompute.py:204-228).
    """
    raw_u16 = _array_arg(raw_u16, ("uint16",), (4,), "precompute_targets")
    h = get_denoiser(device)
    h.set_profile("np", 2)
    return h.targets(raw_u16, offsets, _sigma_scalar(sigma), max_count)


def make_foreground_mask(raw_u16, offset=0.0, k=6.0, dilate=1, device=None):
    """The reference's ``make_foreground_mask(raw, k, dilate)`` (metrics.py:32-61) for
    raw = uint16 patch (or batch) -> float32 - offset: the fallback mask of a patch without
    annotation (data_handling.py:444, :928-929)."""
    return get_denoiser(device).foreground_mask(raw_u16, offset, k, dilate)


def quantize(x, offset_sub=0.0, offset_add=0.0, step=1.0, device=None, truncate=False, z_begin=0):
    """K7; see Denoiser.quantize (step: a scalar or a StepTable)."""
    if isinstance(step, StepTable):
        _step_table_args(step, np.shape(x) if not _is_torch(x) else tuple(x.shape), z_begin)
        return get_denoiser(device).quantize(x, offset_sub, offset_add, step, truncate, z_begin=z_begin)
    return get_denoiser(device).quantize(x, offset_sub, offset_add, step, truncate)


def dequantize(q, step, offset_sub=0.0, offset_add=0.0, z_begin=0, device=None):
    """Inverse of quantize; see Denoiser.dequantize."""
    if isinstance(step, StepTable):
        _step_table_args(step, np.shape(q) if not _is_torch(q) else tuple(q.shape), z_begin)
    return get_denoiser(device).dequantize(q, step, offset_sub, offset_add, z_begin)


def denoise_quantized(vol, sigma, offset_sub=0.0, offset_add=0.0, step=1.0, truncate=False, device=None):
    """Denoise -> background-offset subtract -> (noise-scaled) quantize of one uint16 volume, fused on the device;
    step: a scalar or a StepTable (per-tile steps, e.g. noise_scaled_steps)."""
    if isinstance(step, StepTable):
        shape = np.shape(vol) if not _is_torch(vol) else tuple(vol.shape)
        _step_table_args(step, shape, 0, shape[0])
    return get_denoiser(device).denoise_quantized(vol, sigma, offset_sub, offset_add, step, truncate)


def patch_has_incoherent_segment(labels, raw, min_autocorr=0.4, max_highfreq_frac=0.35, min_segment_voxels=50,
                                 smooth_sigma=1.0, coherence_lag=2, device=None):
    """metrics.patch_has_incoherent_segment (metrics.py:189-260) on the device; same arguments and result."""
    return get_denoiser(device).patch_has_incoherent_segment(labels, raw, min_autocorr, max_highfreq_frac,
                                                             min_segment_voxels, smooth_sigma, coherence_lag)


def noise_scaled_step(sigma_tile, kappa):
    """step = max(1, kappa * sigma_tile) (SURVEY §8a, K7 definition)."""
    return float(max(1.0, float(kappa) * float(sigma_tile)))


def noise_scaled_steps(sigma, kappa, tile):
    """StepTable of float32(noise_scaled_step(sigma, kappa)) per tile: sigma is noise_sigma(x, tile=tile)["sigma"] of
    one volume, (ntz, nty, ntx); a NaN sigma (a tile without usable cells, DESIGN §3.11) gives step 1."""
    s = np.asarray(sigma.detach().cpu().numpy() if _is_torch(sigma) else sigma, dtype=np.float64)
    steps = np.where(np.isnan(s), 1.0, np.maximum(1.0, float(kappa) * s)).astype(np.float32)
    return StepTable(steps, tile)


def tile_stats(x, percentile=1.0, device=None, return_hist=False):
    return get_denoiser(device).tile_stats(x, percentile, return_hist)


def _noise_sigma_args(x, tile):
    """Argument checks of noise_sigma, before any device work: (x, tile tuple or None, tile grid)."""
    x = _array_arg(x, ("uint16",), (3, 4), "noise_sigma")
    if tile is None:
        return x, None, ()
    tile = tuple(int(t) for t in tile)
    if len(tile) != 3 or any(t < 2 or t % 2 for t in tile):
        raise ValueError("tile must be three even sides >= 2, got %r" % (tile,))
    return x, tile, tuple(-(-int(s) // t) for s, t in zip(x.shape[-3:], tile))


def noise_sigma(x, tile=None, device=None, return_hist=False):
    """Noise standard deviation per tile from the MAD of the finest 3-D Haar detail; see Denoiser.noise_sigma.
    Feeds noise_scaled_step and bm4d(z, sigma) with a measured sigma."""
    _noise_sigma_args(x, tile)
    return get_denoiser(device).noise_sigma(x, tile, return_hist)


def noise_sigma_from_hist(hist):
    """{"sigma", "mad", "cells"} of an exact |d| histogram (262141 bins, e.g. the sum of the per-rank histograms of
    noise_sigma(..., return_hist=True)): the same rule as noise_sigma, host arithmetic only."""
    if _is_torch(hist):
        hist = hist.detach().cpu().numpy()
    h = np.ascontiguousarray(hist, dtype=np.int64)
    if h.shape != (_lib.NOISE_HIST_BINS,):
        raise ValueError("hist must have %d bins" % _lib.NOISE_HIST_BINS)
    out = np.empty(2, np.float64)
    cells = np.empty(1, np.int64)
    _lib.check(_lib.load().b4d_noise_sigma_from_hist(h.ctypes.data, out.ctypes.data, out[1:].ctypes.data,
                                                     cells.ctypes.data))
    return {"sigma": out[0], "mad": out[1], "cells": cells[0]}


# --------------------------------------------------------------------------
# Poisson-Gaussian noise (DESIGN §3.12)
# --------------------------------------------------------------------------
class PoissonGaussian(collections.namedtuple("PoissonGaussian", "gain offset read_sigma")):
    """Camera model z = gain * Poisson(lambda) + N(offset, read_sigma^2) of the generalized Anscombe transform:
    gain > 0 (counts per photo-electron), offset (the dark level), read_sigma >= 0 (counts), all finite."""

    __slots__ = ()

    @classmethod
    def from_nlf(cls, a, b, offset):
        """The model of a noise-level function var(z) = a E[z] + b (noise_level_function) and an offset measured
        elsewhere, e.g. tile_stats(x)["offset"]: gain = a, read_sigma = sqrt(max(b + a offset, 0))."""
        a, b, mu = float(a), float(b), float(offset)
        return cls(a, mu, float(np.sqrt(max(b + a * mu, 0.0))))


def default_nlf_edges():
    """0, then 32 * 2^(k/3) for k = 0 .. 33: three bins per octave from 32 to 65536 counts, 34 bins."""
    return np.array([0.0] + [32.0 * 2.0 ** (k / 3.0) for k in range(34)], np.float64)


def _model_c(model):
    """PoissonGaussian (or any (gain, offset, read_sigma)) -> _lib.PgModel; ValueError outside the domain."""
    try:
        gain, offset, read_sigma = (float(v) for v in model)
    except (TypeError, ValueError):
        raise ValueError("model must be a PoissonGaussian (gain, offset, read_sigma), got %r" % (model,))
    if not (np.isfinite(gain) and gain > 0):
        raise ValueError("gain must be positive and finite, got %r" % gain)
    if not np.isfinite(offset):
        raise ValueError("offset must be finite, got %r" % offset)
    if not (np.isfinite(read_sigma) and read_sigma >= 0):
        raise ValueError("read_sigma must be non-negative and finite, got %r" % read_sigma)
    return _lib.PgModel(gain, offset, read_sigma)


def _nlf_args(x, edges, min_cells):
    """Argument checks of noise_level_function, before any device work: (x, edges float64, min_cells)."""
    x = _array_arg(x, ("uint16",), (3, 4), "noise_level_function")
    e = default_nlf_edges() if edges is None else np.ascontiguousarray(edges, dtype=np.float64)
    if e.ndim != 1 or not 2 <= e.size <= _lib.NLF_MAX_BINS + 1:
        raise ValueError("edges must be 2 .. %d values (1 .. %d bins)" % (_lib.NLF_MAX_BINS + 1, _lib.NLF_MAX_BINS))
    if not np.all(np.isfinite(e)) or not np.all(np.diff(e) > 0):
        raise ValueError("edges must be finite and strictly increasing")
    if int(min_cells) < 1:
        raise ValueError("min_cells must be >= 1")
    return x, e, int(min_cells)


def _vst_args(x, sigma, quantize, ndims=(3, 4), what="denoise_vst"):
    """Argument checks of denoise_vst (and its slab forms), before any device work: returns x."""
    if _table_of(quantize) is not None:
        raise NotImplementedError("a step table on the VST path is not implemented")
    x = _array_arg(x, ("uint16",), ndims, what)
    if not (np.isfinite(sigma) and sigma > 0):
        raise ValueError("sigma must be positive and finite, got %r" % (sigma,))
    if quantize is not None and not (3 <= len(quantize) <= 4 and float(quantize[2]) >= 1.0):
        raise ValueError("quantize must be (offset_sub, offset_add, step >= 1[, truncate])")
    return x


def _value_hist(value_hist):
    """The value set of a VST slab (NumPy or torch, host or CUDA) -> C-contiguous int64 NumPy array of 65536 counts;
    ValueError for another length."""
    if _is_torch(value_hist):
        value_hist = value_hist.detach().cpu().numpy()
    h = np.ascontiguousarray(value_hist, dtype=np.int64)
    if h.shape != (65536,):
        raise ValueError("value_hist must hold 65536 counts (one per uint16 value), got shape %r" % (h.shape,))
    return h


def noise_level_function(x, edges=None, min_cells=256, device=None):
    """Noise-level function of Poisson-Gaussian counts; see Denoiser.noise_level_function."""
    _nlf_args(x, edges, min_cells)
    return get_denoiser(device).noise_level_function(x, edges, min_cells)


def gat_forward(x, model, device=None):
    """Generalized Anscombe transform; see Denoiser.gat_forward."""
    _array_arg(x, ("uint16",), None, "gat_forward")
    _model_c(model)
    return get_denoiser(device).gat_forward(x, model)


def gat_inverse(y, model, device=None):
    """Inverse of gat_forward; see Denoiser.gat_inverse."""
    _array_arg(y, ("float32",), None, "gat_inverse")
    _model_c(model)
    return get_denoiser(device).gat_inverse(y, model)


def denoise_vst(x, model, sigma=1.0, quantize=None, device=None):
    """Denoise Poisson-Gaussian uint16 counts through the GAT; see Denoiser.denoise_vst."""
    _vst_args(x, sigma, quantize)
    _model_c(model)
    return get_denoiser(device).denoise_vst(x, model, sigma, quantize)
