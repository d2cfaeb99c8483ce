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
import ctypes
import enum
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

    def debug_accumulators(self, n):
        """(numq, wmap) int64 arrays: the fixed-point aggregation state the last filter stage of the last
        single-volume call left on the device (b4d_debug_accumulators; diagnostics for the parity tests)."""
        numq = np.empty(n, dtype=np.int64)
        wmap = np.empty(n, dtype=np.int64)
        _lib.check(self.lib.b4d_debug_accumulators(self._h, numq.ctypes.data_as(ctypes.c_void_p),
                                                   wmap.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(n)))
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
        _lib.check(self.lib.b4d_set_noise_model(self._h, a.ctypes.data_as(ctypes.c_void_p),
                                                b.ctypes.data_as(ctypes.c_void_p)))

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
        _lib.check(
            fn(
                self._h,
                ctypes.c_void_p(in_ptr),
                ctypes.c_int64(n),
                _lib.shape3(shape),
                ctypes.c_float(sigma),
                ctypes.c_void_p(out_ptr),
                int(in_dev),
                int(out_dev),
            )
        )

    # ---- array level ---------------------------------------------------------
    def denoise(self, z, sigma):
        """(D,H,W) or (N,D,H,W); uint16 or float32; NumPy or torch -> float32."""
        if _is_torch(z):
            import torch

            if z.dtype not in (torch.uint16, torch.float32):
                raise ValueError("torch input must be uint16 or float32, got %s" % z.dtype)
            zc = z.contiguous()
            if zc.ndim not in (3, 4):
                raise ValueError("expected a 3-D volume or a 4-D batch, got %d-D" % zc.ndim)
            n = zc.shape[0] if zc.ndim == 4 else 1
            on_dev = zc.is_cuda
            if on_dev and zc.device.index != self.device:
                raise ValueError("tensor lives on cuda:%s, handle on cuda:%d" % (zc.device.index, self.device))
            out = torch.empty(zc.shape, dtype=torch.float32, device=zc.device)
            if on_dev:
                torch.cuda.current_stream(zc.device).synchronize()
            self.denoise_ptr(
                zc.data_ptr(),
                np.uint16 if zc.dtype == torch.uint16 else np.float32,
                n,
                tuple(zc.shape[-3:]),
                sigma,
                out.data_ptr(),
                on_dev,
                on_dev,
            )
            return out
        z = np.asarray(z)
        if z.ndim not in (3, 4):
            raise ValueError("expected a 3-D volume or a 4-D batch, got %d-D" % z.ndim)
        zc = np.ascontiguousarray(z)
        n = zc.shape[0] if zc.ndim == 4 else 1
        out = np.empty(zc.shape, dtype=np.float32)
        self.denoise_ptr(zc.ctypes.data, zc.dtype.type, n, zc.shape[-3:], sigma, out.ctypes.data, 0, 0)
        return out

    def targets(self, raw_u16, offsets, sigma, max_count=65535.0, raw_out=None, teacher_out=None):
        """(N,D,H,W) uint16 patches + per-patch offsets -> (raw, teacher) float32 in one call
        (b4d_targets_u16: subtraction, BM4D and clip all on the device).  `raw_out` / `teacher_out`
        may be preallocated C-contiguous float32 arrays (e.g. the cache's memmaps)."""
        zc = np.ascontiguousarray(raw_u16)
        if zc.ndim != 4 or zc.dtype != np.uint16:
            raise ValueError("raw_u16 must be (N, D, H, W) uint16")
        off = np.ascontiguousarray(np.broadcast_to(np.asarray(offsets, dtype=np.float32), (zc.shape[0],)))
        outs = []
        for o in (raw_out, teacher_out):
            if o is None:
                o = np.empty(zc.shape, dtype=np.float32)
            elif o.shape != zc.shape or o.dtype != np.float32 or not o.flags.c_contiguous:
                raise ValueError("output must be a C-contiguous float32 array of shape %r" % (zc.shape,))
            outs.append(o)
        _lib.check(
            self.lib.b4d_targets_u16(
                self._h,
                ctypes.c_void_p(zc.ctypes.data),
                ctypes.c_int64(zc.shape[0]),
                _lib.shape3(zc.shape[1:]),
                ctypes.c_void_p(off.ctypes.data),
                ctypes.c_float(sigma),
                ctypes.c_float(max_count),
                ctypes.c_void_p(outs[0].ctypes.data),
                ctypes.c_void_p(outs[1].ctypes.data),
                0,
                0,
            )
        )
        return outs[0], outs[1]

    def denoise_slab(self, slab, z_begin, z_total, own_begin, own_end, sigma, out=None, quantize=None):
        """One z-slab (uint16, with halos) of a larger volume -> float32 owned planes.
        `out` (NumPy path only) receives the result in place, e.g. a pinned buffer.
        quantize = (offset_sub, offset_add, step[, truncate]): the fused denoise -> offset -> quantize path, the
        result is the uint16 volume K7 would give on the float32 output (2 bytes per voxel leave the device)."""
        odt_np, odt_t = (np.float32, "float32") if quantize is None else (np.uint16, "uint16")
        if _is_torch(slab):
            import torch

            sc = slab.contiguous()
            if sc.dtype != torch.uint16 or sc.ndim != 3:
                raise ValueError("slab must be a 3-D uint16 tensor")
            out = torch.empty((own_end - own_begin,) + tuple(sc.shape[1:]), dtype=getattr(torch, odt_t), device=sc.device)
            on_dev = sc.is_cuda
            if on_dev:
                torch.cuda.current_stream(sc.device).synchronize()
            in_ptr, out_ptr, shape = sc.data_ptr(), out.data_ptr(), tuple(sc.shape)
        else:
            sc = np.ascontiguousarray(slab)
            if sc.dtype != np.uint16 or sc.ndim != 3:
                raise ValueError("slab must be a 3-D uint16 array")
            oshape = (own_end - own_begin,) + sc.shape[1:]
            if out is None:
                out = np.empty(oshape, dtype=odt_np)
            elif out.shape != oshape or out.dtype != odt_np or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous %s array of shape %r" % (odt_t, oshape))
            on_dev = False
            in_ptr, out_ptr, shape = sc.ctypes.data, out.ctypes.data, sc.shape
        if quantize is not None:
            q = tuple(quantize) + (False,) * (4 - len(quantize))
            _lib.check(
                self.lib.b4d_denoise_slab_q16_u16(
                    self._h, ctypes.c_void_p(in_ptr), _lib.shape3(shape), ctypes.c_int64(z_begin),
                    ctypes.c_int64(z_total), ctypes.c_int64(own_begin), ctypes.c_int64(own_end), ctypes.c_float(sigma),
                    ctypes.c_float(q[0]), ctypes.c_float(q[1]), ctypes.c_float(q[2]), int(bool(q[3])),
                    ctypes.c_void_p(out_ptr), int(on_dev), int(on_dev),
                )
            )
            return out
        _lib.check(
            self.lib.b4d_denoise_slab_u16(
                self._h,
                ctypes.c_void_p(in_ptr),
                _lib.shape3(shape),
                ctypes.c_int64(z_begin),
                ctypes.c_int64(z_total),
                ctypes.c_int64(own_begin),
                ctypes.c_int64(own_end),
                ctypes.c_float(sigma),
                ctypes.c_void_p(out_ptr),
                int(on_dev),
                int(on_dev),
            )
        )
        return out

    # ---- the slab in two calls, for one neighbour exchange between the stages ----
    def slab_stage1(self, slab, z_begin, z_total, sigma):
        """Stage 1 on a uint16 slab (NumPy or torch); the basic estimate stays on the device."""
        if _is_torch(slab):
            import torch

            sc = slab.contiguous()
            if sc.dtype != torch.uint16 or sc.ndim != 3:
                raise ValueError("slab must be a 3-D uint16 tensor")
            on_dev = sc.is_cuda
            if on_dev:
                torch.cuda.current_stream(sc.device).synchronize()
            ptr, shape = sc.data_ptr(), tuple(sc.shape)
        else:
            sc = np.ascontiguousarray(slab)
            if sc.dtype != np.uint16 or sc.ndim != 3:
                raise ValueError("slab must be a 3-D uint16 array")
            on_dev, ptr, shape = False, sc.ctypes.data, sc.shape
        self._slab_shape = tuple(int(v) for v in shape)
        _lib.check(
            self.lib.b4d_slab_stage1_u16(self._h, ctypes.c_void_p(ptr), _lib.shape3(shape), ctypes.c_int64(z_begin),
                                         ctypes.c_int64(z_total), ctypes.c_float(sigma), int(on_dev))
        )

    def slab_basic(self, plane0, nplanes, device=None):
        """Planes [plane0, plane0 + nplanes) (slab-local) of the basic estimate: a torch CUDA
        tensor when `device` is given, else a NumPy array."""
        shape = (int(nplanes),) + self._slab_shape[1:]
        if device is not None:
            import torch

            buf = torch.empty(shape, dtype=torch.float32, device=device)
            ptr, on_dev = buf.data_ptr(), True
        else:
            buf = np.empty(shape, dtype=np.float32)
            ptr, on_dev = buf.ctypes.data, False
        if nplanes:
            _lib.check(self.lib.b4d_slab_basic_planes(self._h, ctypes.c_int64(plane0), ctypes.c_int64(nplanes),
                                                      ctypes.c_void_p(ptr), 0, int(on_dev)))
        return buf

    def slab_set_basic(self, plane0, planes):
        """Overwrite planes of the basic estimate (the neighbour's exact halo planes)."""
        if _is_torch(planes):
            import torch

            pc = planes.contiguous()
            if pc.dtype != torch.float32:
                raise ValueError("planes must be float32")
            if pc.is_cuda:
                torch.cuda.current_stream(pc.device).synchronize()
            ptr, on_dev, n = pc.data_ptr(), pc.is_cuda, pc.shape[0]
        else:
            pc = np.ascontiguousarray(planes, dtype=np.float32)
            ptr, on_dev, n = pc.ctypes.data, False, pc.shape[0]
        if tuple(pc.shape[1:]) != self._slab_shape[1:]:
            raise ValueError("planes must have the slab's (H, W)")
        if n:
            _lib.check(self.lib.b4d_slab_basic_planes(self._h, ctypes.c_int64(plane0), ctypes.c_int64(n),
                                                      ctypes.c_void_p(ptr), 1, int(on_dev)))

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
        _lib.check(self.lib.b4d_slab_stage2_begin(self._h, ctypes.c_int64(own_begin), ctypes.c_int64(own_end)))

    def slab_stage2(self, own_begin, own_end, out=None, device=None, quantize=None):
        """Stage 2 on the completed basic estimate -> float32 owned planes (NumPy, or torch on
        `device`; `out` may be a preallocated NumPy array, e.g. pinned).  quantize = (offset_sub, offset_add,
        step[, truncate]): uint16 output of the fused quantizer instead (see denoise_slab)."""
        oshape = (int(own_end - own_begin),) + self._slab_shape[1:]
        odt_np, odt_t = (np.float32, "float32") if quantize is None else (np.uint16, "uint16")
        if device is not None:
            import torch

            out = torch.empty(oshape, dtype=getattr(torch, odt_t), device=device)
            ptr, on_dev = out.data_ptr(), True
        else:
            if out is None:
                out = np.empty(oshape, dtype=odt_np)
            elif out.shape != oshape or out.dtype != odt_np or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous %s array of shape %r" % (odt_t, oshape))
            ptr, on_dev = out.ctypes.data, False
        if quantize is not None:
            q = tuple(quantize) + (False,) * (4 - len(quantize))
            _lib.check(self.lib.b4d_slab_stage2_q16(self._h, ctypes.c_int64(own_begin), ctypes.c_int64(own_end),
                                                    ctypes.c_float(q[0]), ctypes.c_float(q[1]), ctypes.c_float(q[2]),
                                                    int(bool(q[3])), ctypes.c_void_p(ptr), int(on_dev)))
            return out
        _lib.check(self.lib.b4d_slab_stage2(self._h, ctypes.c_int64(own_begin), ctypes.c_int64(own_end),
                                            ctypes.c_void_p(ptr), int(on_dev)))
        return out

    def denoise_quantized(self, vol, sigma, offset_sub=0.0, offset_add=0.0, step=1.0, truncate=False, out=None):
        """denoise -> offset -> quantize of one uint16 volume in one call (b4d_denoise_q16_u16): the uint16 volume
        `quantize(denoise(vol, sigma), offset_sub, offset_add, step, truncate)` would give, bit for bit."""
        D = int(vol.shape[0])
        return self.denoise_slab(vol, 0, D, 0, D, sigma, out=out, quantize=(offset_sub, offset_add, step, truncate))

    def match_stage1(self, vol, sigma):
        """Instrumented stage-1 matcher: (idx[R,K] int32, ssd[R,K] uint64, count[R] int32)."""
        vol = np.ascontiguousarray(vol)
        if vol.dtype != np.uint16 or vol.ndim != 3:
            raise ValueError("match_stage1 expects a 3-D uint16 array")
        shape = _lib.shape3(vol.shape)
        R = self.lib.b4d_num_refs(shape)
        K = int(self.profile.max_stack_size_ht)
        idx = np.empty((R, K), dtype=np.int32)
        ssd = np.empty((R, K), dtype=np.uint64)
        cnt = np.empty((R,), dtype=np.int32)
        _lib.check(
            self.lib.b4d_match_stage1(
                self._h,
                ctypes.c_void_p(vol.ctypes.data),
                shape,
                ctypes.c_float(sigma),
                ctypes.c_void_p(idx.ctypes.data),
                ctypes.c_void_p(ssd.ctypes.data),
                ctypes.c_void_p(cnt.ctypes.data),
            )
        )
        return idx, ssd, cnt

    def quantize(self, x, offset_sub=0.0, offset_add=0.0, step=1.0, truncate=False):
        """K7: rint(clip((x - offset_sub + offset_add)/step, 0, 65535/step)) -> uint16.
        truncate=True: the evaluator's variant, np.maximum(v, 0).astype(int) cast to uint16 (evaluate.py:202,
        utils/img_util.py:420-423): toward zero, no upper clip, wrapping modulo 2^16."""
        if _is_torch(x):
            import torch

            xc = x.contiguous()
            if xc.dtype != torch.float32:
                raise ValueError("quantize expects float32")
            out = torch.empty(xc.shape, dtype=torch.uint16, device=xc.device)
            on_dev = xc.is_cuda
            if on_dev:
                torch.cuda.current_stream(xc.device).synchronize()
            in_ptr, out_ptr, n = xc.data_ptr(), out.data_ptr(), xc.numel()
        else:
            xc = np.ascontiguousarray(x, dtype=np.float32)
            out = np.empty(xc.shape, dtype=np.uint16)
            on_dev = False
            in_ptr, out_ptr, n = xc.ctypes.data, out.ctypes.data, xc.size
        fn = self.lib.b4d_quantize_trunc_u16 if truncate else self.lib.b4d_quantize_u16
        _lib.check(
            fn(
                self._h,
                ctypes.c_void_p(in_ptr),
                ctypes.c_int64(n),
                ctypes.c_float(offset_sub),
                ctypes.c_float(offset_add),
                ctypes.c_float(step),
                ctypes.c_void_p(out_ptr),
                int(on_dev),
                int(on_dev),
            )
        )
        return out

    def set_pass_voxels(self, voxels):
        """Voxels per pass (scratch ~45 B each; 0 = default 1.25 Gi).  A uint16 volume larger than a
        pass is denoised as consecutive z-slabs with halos; the result does not change."""
        _lib.check(self.lib.b4d_set_pass_voxels(self._h, ctypes.c_int64(int(voxels))))

    def set_pipeline_min_voxels(self, voxels):
        """Volume size from which host transfers are pipelined against the kernels (default 2^26)."""
        _lib.check(self.lib.b4d_set_pipeline_min_voxels(self._h, ctypes.c_int64(int(voxels))))

    def foreground_mask(self, raw_u16, offsets=0.0, k=6.0, dilate=1):
        """make_foreground_mask (metrics.py:32-61) of uint16 patches after the offset subtraction
        (data_handling.py:353-354): (D,H,W) or (N,D,H,W) uint16 -> bool mask of the same shape."""
        zc = np.ascontiguousarray(raw_u16)
        if zc.dtype != np.uint16 or zc.ndim not in (3, 4):
            raise ValueError("raw_u16 must be a uint16 volume or a (N, D, H, W) batch")
        n = zc.shape[0] if zc.ndim == 4 else 1
        off = np.ascontiguousarray(np.broadcast_to(np.asarray(offsets, dtype=np.float32), (n,)))
        out = np.empty(zc.shape, dtype=np.uint8)
        _lib.check(
            self.lib.b4d_foreground_mask_u16(
                self._h,
                ctypes.c_void_p(zc.ctypes.data),
                ctypes.c_int64(n),
                _lib.shape3(zc.shape[-3:]),
                ctypes.c_void_p(off.ctypes.data),
                ctypes.c_float(k),
                ctypes.c_int(int(dilate)),
                ctypes.c_void_p(out.ctypes.data),
                0,
                0,
            )
        )
        return out.view(np.bool_)

    def chunk_shuffle(self, x, chunk=(64, 64, 64), want_bytes=True, want_hist=True):
        """K9: C-order chunk gather + Blosc 2-byte shuffle of a uint16 volume, plus per-piece byte
        histograms [pieces, 2, 256] (uint32).  Returns (bytes or None, hist or None)."""
        if len(chunk) != 3:
            raise ValueError("chunk must have three entries")
        if not (want_bytes or want_hist):
            raise ValueError("nothing requested")
        torch_in = _is_torch(x)
        if torch_in:
            import torch

            xc = x.contiguous()
            if xc.dtype != torch.uint16 or xc.ndim != 3:
                raise ValueError("chunk_shuffle expects a 3-D uint16 volume")
            on_dev = xc.is_cuda
            if on_dev:
                torch.cuda.current_stream(xc.device).synchronize()
            shape, in_ptr = tuple(xc.shape), xc.data_ptr()
        else:
            xc = np.ascontiguousarray(x)
            if xc.dtype != np.uint16 or xc.ndim != 3:
                raise ValueError("chunk_shuffle expects a 3-D uint16 volume")
            on_dev = False
            shape, in_ptr = xc.shape, xc.ctypes.data
        npieces = 1
        for s_, c_ in zip(shape, chunk):
            if int(c_) < 1:
                raise ValueError("chunk sides must be >= 1")
            npieces *= -(-int(s_) // int(c_))
        nvox = int(shape[0]) * int(shape[1]) * int(shape[2])
        out = hist = None
        out_ptr = hist_ptr = None
        if on_dev:
            if want_bytes:
                out = torch.empty(2 * nvox, dtype=torch.uint8, device=xc.device)
                out_ptr = out.data_ptr()
            if want_hist:
                hist = torch.empty((npieces, 2, 256), dtype=torch.int32, device=xc.device)
                hist_ptr = hist.data_ptr()
        else:
            if want_bytes:
                out = np.empty(2 * nvox, dtype=np.uint8)
                out_ptr = out.ctypes.data
            if want_hist:
                hist = np.empty((npieces, 2, 256), dtype=np.uint32)
                hist_ptr = hist.ctypes.data
        _lib.check(
            self.lib.b4d_chunk_shuffle_u16(
                self._h,
                ctypes.c_void_p(in_ptr),
                _lib.shape3(shape),
                _lib.shape3(chunk),
                ctypes.c_void_p(out_ptr),
                ctypes.c_void_p(hist_ptr),
                int(on_dev),
                int(on_dev),
            )
        )
        if torch_in and not on_dev:
            import torch

            out = torch.from_numpy(out) if out is not None else None
            hist = torch.from_numpy(hist.view(np.int32)) if hist is not None else None
        return out, hist

    def tile_stats(self, x, percentile=1.0, return_hist=False):
        """K8: offset percentile over non-zero voxels + median / MAD sigma of a uint16 tile."""
        if _is_torch(x):
            import torch

            xc = x.contiguous()
            if xc.dtype != torch.uint16:
                raise ValueError("tile_stats expects uint16")
            on_dev = xc.is_cuda
            if on_dev:
                torch.cuda.current_stream(xc.device).synchronize()
            in_ptr, n = xc.data_ptr(), xc.numel()
        else:
            xc = np.ascontiguousarray(x)
            if xc.dtype != np.uint16:
                raise ValueError("tile_stats expects uint16")
            on_dev = False
            in_ptr, n = xc.ctypes.data, xc.size
        st = _lib.Stats()
        hist = np.empty(65536, dtype=np.int64) if return_hist else None
        _lib.check(
            self.lib.b4d_tile_stats(
                self._h,
                ctypes.c_void_p(in_ptr),
                ctypes.c_int64(n),
                ctypes.c_double(percentile),
                ctypes.byref(st),
                ctypes.c_void_p(hist.ctypes.data) if return_hist else None,
                int(on_dev),
            )
        )
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
        x, shape, tile, grid = _noise_sigma_args(x, tile)
        if _is_torch(x):
            import torch

            xc = x.contiguous()
            on_dev = xc.is_cuda
            if on_dev:
                torch.cuda.current_stream(xc.device).synchronize()
            in_ptr = xc.data_ptr()
        else:
            xc = np.ascontiguousarray(x)
            on_dev = False
            in_ptr = xc.ctypes.data
        n = 1 if len(shape) == 3 else shape[0]
        out_shape = (() if len(shape) == 3 else (n,)) + grid
        sigma = np.empty(out_shape, np.float64)
        mad = np.empty(out_shape, np.float64)
        cells = np.empty(out_shape, np.int64)
        hist = np.empty(_lib.NOISE_HIST_BINS, np.int64) if return_hist else None
        _lib.check(
            self.lib.b4d_noise_sigma_u16(
                self._h, in_ptr, n, _lib.shape3(shape[-3:]), _lib.shape3(tile) if tile is not None else None,
                sigma.ctypes.data, mad.ctypes.data, cells.ctypes.data, hist.ctypes.data if return_hist else None,
                int(on_dev),
            )
        )
        d = {"sigma": sigma[()], "mad": mad[()], "cells": cells[()]}
        return (d, hist) if return_hist else d

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
                self._h, x.ctypes.data_as(ctypes.c_void_p), lab.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(n),
                _lib.shape3(shape), ctypes.c_double(min_autocorr), ctypes.c_double(max_highfreq_frac),
                ctypes.c_int64(min_segment_voxels), ctypes.c_double(smooth_sigma), ctypes.c_int(coherence_lag),
                reject.ctypes.data_as(ctypes.c_void_p), seg, ctypes.c_int64(max_segments),
                cnt.ctypes.data_as(ctypes.c_void_p), 0,
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
    raw_u16 = np.asarray(raw_u16)
    if raw_u16.ndim != 4 or raw_u16.dtype != np.uint16:
        raise ValueError("raw_u16 must be (N, D, H, W) uint16")
    h = get_denoiser(device)
    h.set_profile("np", 2)
    return h.targets(raw_u16, offsets, _sigma_scalar(sigma), max_count)


def make_foreground_mask(raw_u16, offset=0.0, k=6.0, dilate=1, device=None):
    """The reference's ``make_foreground_mask(raw, k, dilate)`` (metrics.py:32-61) for
    raw = uint16 patch (or batch) -> float32 - offset: the fallback mask of a patch without
    annotation (data_handling.py:444, :928-929)."""
    return get_denoiser(device).foreground_mask(raw_u16, offset, k, dilate)


def quantize(x, offset_sub=0.0, offset_add=0.0, step=1.0, device=None, truncate=False):
    return get_denoiser(device).quantize(x, offset_sub, offset_add, step, truncate)


def denoise_quantized(vol, sigma, offset_sub=0.0, offset_add=0.0, step=1.0, truncate=False, device=None):
    """Denoise -> background-offset subtract -> (noise-scaled) quantize of one uint16 volume, fused on the device."""
    return get_denoiser(device).denoise_quantized(vol, sigma, offset_sub, offset_add, step, truncate)


def patch_has_incoherent_segment(labels, raw, min_autocorr=0.4, max_highfreq_frac=0.35, min_segment_voxels=50,
                                 smooth_sigma=1.0, coherence_lag=2, device=None):
    """metrics.patch_has_incoherent_segment (metrics.py:189-260) on the device; same arguments and result."""
    return get_denoiser(device).patch_has_incoherent_segment(labels, raw, min_autocorr, max_highfreq_frac,
                                                             min_segment_voxels, smooth_sigma, coherence_lag)


def noise_scaled_step(sigma_tile, kappa):
    """step = max(1, kappa * sigma_tile) (SURVEY §8a, K7 definition)."""
    return float(max(1.0, float(kappa) * float(sigma_tile)))


def tile_stats(x, percentile=1.0, device=None, return_hist=False):
    return get_denoiser(device).tile_stats(x, percentile, return_hist)


def _noise_sigma_args(x, tile):
    """Argument checks of noise_sigma, before any device work: (x, shape, tile tuple or None, tile grid)."""
    if _is_torch(x):
        import torch

        ok = x.dtype == torch.uint16
        shape = tuple(int(s) for s in x.shape)
    else:
        x = np.asarray(x)
        ok = x.dtype == np.uint16
        shape = x.shape
    if not ok:
        raise ValueError("noise_sigma expects uint16, got %s" % (x.dtype,))
    if len(shape) not in (3, 4):
        raise ValueError("noise_sigma expects a 3-D volume or a 4-D batch, got %d-D" % len(shape))
    if tile is None:
        return x, shape, None, ()
    tile = tuple(int(t) for t in tile)
    if len(tile) != 3 or any(t < 2 or t % 2 for t in tile):
        raise ValueError("tile must be three even sides >= 2, got %r" % (tile,))
    return x, shape, tile, tuple(-(-s // t) for s, t in zip(shape[-3:], tile))


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
