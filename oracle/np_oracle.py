"""CPU ORACLE (Python side).  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product never does.

Two things live here:

1. NumPy restatements of the steps that DO exist in the reference tree, each
   following the cited lines (paths under /root/reference/src/
   aind_exaspim_image_compression/).  They are pinned against the imported
   reference by ``tests/golden/make_golden.py`` -> ``tests/golden/*.npz``.
2. A ctypes loader for ``oracle/liboracle.so`` (b4d_oracle.cpp), the C++
   restatement of the BM4D algorithm itself.  PARITY UNPINNED for that part:
   the reference's BM4D is the closed wheel bm4d==4.2.5, absent everywhere.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
MAX_COUNT = 65535.0  # transforms.py:92, :108


# --------------------------------------------------------------------------
# 1. steps present in the reference tree
# --------------------------------------------------------------------------
def read_counts(raw_u16, offset):
    """uint16 -> float32, subtract the per-brain scalar (data_handling.py:353-354)."""
    raw = np.asarray(raw_u16).astype(np.float32)
    return raw - offset


def clip_teacher(teacher, max_count=MAX_COUNT):
    """np.clip(teacher, 0, transform.max_count) (data_handling.py:333, :927)."""
    return np.clip(teacher, 0, max_count)


def quantize_reference(counts, offset_add=0.0, max_count=MAX_COUNT):
    """Pedestal restore + clip + rint + uint16 (transforms.py:403-411, :150-152).

    ``counts`` float32; a float32 array plus a Python float stays float32, clip
    and rint keep float32, rint is round-half-to-even.
    """
    counts = np.asarray(counts, dtype=np.float32)
    if offset_add != 0.0:
        counts = counts + offset_add  # transforms.py:405
    counts = np.clip(counts, 0, max_count)  # transforms.py:410
    return np.rint(counts).astype(np.uint16)  # transforms.py:411


def quantize_noise_scaled(x, offset_sub=0.0, offset_add=0.0, step=1.0):
    """K7 contract (SURVEY §8a row Q / DESIGN.md §3.7), float32 throughout:

    q = rint(clip((x - offset_sub + offset_add) / step, 0, 65535 / step)) -> uint16
    """
    f32 = np.float32
    v = (np.asarray(x, dtype=f32) - f32(offset_sub)) + f32(offset_add)
    if f32(step) != f32(1.0):
        v = v / f32(step)
    hi = f32(65535.0) / f32(step)
    v = np.minimum(np.maximum(v, f32(0.0)), hi)
    return np.rint(v).astype(np.uint16)


def quantize_truncating(x):
    """np.maximum(x, 0).astype(int) (evaluate.py:202) then the uint16 cast of
    compute_cratio (utils/img_util.py:420-423)."""
    return np.ascontiguousarray(np.maximum(x, 0).astype(int), dtype=np.uint16)


def make_foreground_mask_reference(raw, k=6.0, dilate=1):
    """Intensity foreground mask (metrics.py:54-61): median + k * (1.4826 * MAD) threshold in float32,
    then `dilate` iterations of binary dilation with the 6-neighbour structuring element and border
    value 0 (what scipy.ndimage.binary_dilation does by default), written with array shifts."""
    raw = np.asarray(raw, dtype=np.float32)
    med = np.median(raw)
    mad = np.median(np.abs(raw - med)) + 1e-6
    sigma = 1.4826 * mad
    mask = raw > (med + k * sigma)
    for _ in range(int(dilate)):
        grown = mask.copy()
        for ax in range(mask.ndim):
            lo = [slice(None)] * mask.ndim
            hi = [slice(None)] * mask.ndim
            lo[ax], hi[ax] = slice(0, -1), slice(1, None)
            grown[tuple(lo)] |= mask[tuple(hi)]
            grown[tuple(hi)] |= mask[tuple(lo)]
        mask = grown
    return mask


def coherence_scores_reference(labels, raw, smooth_sigma=1.0, lag=2):
    """Per-segment (voxels, lag autocorrelation, high-frequency energy fraction) the way the sampler's gate
    computes them: local_autocorr (metrics.py:96-112), highfreq_energy_fraction (:148-155) with the Gaussian
    smooth of the whole patch (:247-248), all float64.  Returns {label: (voxels, autocorr, highfreq)}."""
    from scipy import ndimage

    labels = np.asarray(labels)
    raw = np.asarray(raw, dtype=np.float64)
    smooth = ndimage.gaussian_filter(raw, sigma=smooth_sigma)
    out = {}
    for lid in np.unique(labels[labels > 0]):
        seg = labels == lid
        vals = []
        for ax in range(raw.ndim):
            lo = [slice(None)] * raw.ndim
            hi = [slice(None)] * raw.ndim
            lo[ax], hi[ax] = slice(0, -lag), slice(lag, None)
            sel = seg[tuple(lo)] & seg[tuple(hi)]
            if sel.sum() < 2:
                continue
            x, y = raw[tuple(lo)][sel], raw[tuple(hi)][sel]
            if x.std() < 1e-6 or y.std() < 1e-6:
                continue
            vals.append(float(np.corrcoef(x, y)[0, 1]))
        ac = float(np.mean(vals)) if vals else 1.0
        v = raw[seg]
        hf = 0.0 if v.var() < 1e-12 else float((raw - smooth)[seg].var() / v.var())
        out[int(lid)] = (int(seg.sum()), ac, hf)
    return out


def patch_has_incoherent_segment_reference(labels, raw, min_autocorr=0.4, max_highfreq_frac=0.35,
                                           min_segment_voxels=50, smooth_sigma=1.0, coherence_lag=2):
    """The gate's decision (metrics.py:241-260) from the scores above."""
    sc = coherence_scores_reference(labels, raw, smooth_sigma, coherence_lag)
    return any(n >= min_segment_voxels and ac < min_autocorr and hf > max_highfreq_frac for n, ac, hf in sc.values())


def chunk_shuffle_reference(img, patch_shape=(64, 64, 64)):
    """The chunk loop of compute_cratio (utils/img_util.py:427-438) with Blosc's byte shuffle for
    2-byte items applied to each piece instead of the codec call: returns (bytes of all pieces back
    to back — low bytes then high bytes per piece —, hist[pieces, 2, 256])."""
    img = np.ascontiguousarray(img, dtype=np.uint16)  # img_util.py:423
    parts, hists = [], []
    z = [range(0, s, c) for s, c in zip(img.shape, patch_shape)]
    for z0 in z[0]:
        for z1 in z[1]:
            for z2 in z[2]:
                piece = np.ascontiguousarray(
                    img[z0 : z0 + patch_shape[0], z1 : z1 + patch_shape[1], z2 : z2 + patch_shape[2]]
                )
                by = piece.reshape(-1).view(np.uint8).reshape(-1, 2)  # little endian: [:, 0] low, [:, 1] high
                lo, hi = np.ascontiguousarray(by[:, 0]), np.ascontiguousarray(by[:, 1])
                parts += [lo, hi]
                hists.append([np.bincount(lo, minlength=256), np.bincount(hi, minlength=256)])
    return np.concatenate(parts), np.asarray(hists, dtype=np.uint32)


def estimate_offset(sample, percentile=1.0, ignore_zeros=True):
    """Low percentile over non-zero voxels (transforms.py:433-438)."""
    sample = np.asarray(sample, dtype=np.float32).reshape(-1)
    if ignore_zeros:
        nonzero = sample[sample > 0]
        if nonzero.size:
            sample = nonzero
    return float(np.percentile(sample, percentile))


def robust_sigma(raw):
    """median / MAD noise statistic (metrics.py:54-57). Returns (med, mad, sigma)."""
    raw = np.asarray(raw, dtype=np.float32)
    med = np.median(raw)
    mad = np.median(np.abs(raw - med)) + 1e-6
    sigma = 1.4826 * mad
    return float(med), float(mad), float(sigma)


# --------------------------------------------------------------------------
# 2. liboracle.so (C++ restatement of BM4D)
# --------------------------------------------------------------------------
class Profile(ctypes.Structure):
    _fields_ = [
        ("abi", ctypes.c_int32),
        ("block", ctypes.c_int32),
        ("step", ctypes.c_int32),
        ("search_ht", ctypes.c_int32),
        ("search_wie", ctypes.c_int32),
        ("k_ht", ctypes.c_int32),
        ("k_wie", ctypes.c_int32),
        ("stages", ctypes.c_int32),
        ("deterministic", ctypes.c_int32),
        ("reserved0", ctypes.c_int32),
        ("tau_ht", ctypes.c_float),
        ("tau_wie", ctypes.c_float),
        ("lambda_ht", ctypes.c_float),
        ("kaiser_beta", ctypes.c_float),
    ]


_lib = None


def lib_path():
    return os.path.join(_HERE, "liboracle.so")


def load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(lib_path())
        lib.b4d_last_error.restype = ctypes.c_char_p
        lib.b4d_num_refs.restype = ctypes.c_int64
        _lib = lib
    return _lib


def set_threads(n=0):
    """Set the oracle's OpenMP team size (n <= 0: leave it) and return the size in effect."""
    return int(load().b4d_oracle_set_threads(int(n)))


def _check(rc):
    if rc != 0:
        raise RuntimeError("oracle: %s (status %d)" % (load().b4d_last_error().decode(), rc))


def default_profile(**overrides):
    p = Profile()
    load().b4d_default_profile(ctypes.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def match_map(z, sigma):
    """(integral, scale, centre) of the matching map the oracle matches float32 data z with at this sigma
    (DESIGN §3.1): integral-count map or not, its power-of-two scale, and the DC level c0 subtracted first (0: none)."""
    z = np.ascontiguousarray(z, dtype=np.float32)
    integral, scale, centre = ctypes.c_int(), ctypes.c_float(), ctypes.c_float()
    _check(load().b4d_oracle_match_map(z.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(z.size), ctypes.c_float(sigma),
                                       ctypes.byref(integral), ctypes.byref(scale), ctypes.byref(centre)))
    return bool(integral.value), float(scale.value), float(centre.value)


class Oracle:
    """arith='f64' (plain restatement) or 'mirror' (float32, CUDA operation order)."""

    def __init__(self, arith="f64", **profile):
        lib = load()
        self.profile = default_profile(**profile)
        self._h = ctypes.c_void_p()
        _check(lib.b4d_create(0, ctypes.byref(self.profile), ctypes.byref(self._h)))
        _check(lib.b4d_oracle_set_arith(self._h, {"mirror": 0, "f64": 1}[arith]))

    def close(self):
        if self._h:
            load().b4d_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _shape3(shape):
        return (ctypes.c_int64 * 3)(*[int(s) for s in shape])

    def denoise(self, z, sigma):
        """z: (D,H,W) or (N,D,H,W), uint16 or float32 -> float32 same shape."""
        z = np.ascontiguousarray(z)
        batched = z.ndim == 4
        n = z.shape[0] if batched else 1
        shape = z.shape[-3:]
        out = np.empty(z.shape, dtype=np.float32)
        lib = load()
        if z.dtype == np.uint16:
            fn = lib.b4d_denoise_u16
        elif z.dtype == np.float32:
            fn = lib.b4d_denoise_f32
        else:
            raise ValueError("dtype must be uint16 or float32")
        _check(
            fn(
                self._h,
                z.ctypes.data_as(ctypes.c_void_p),
                ctypes.c_int64(n),
                self._shape3(shape),
                ctypes.c_float(sigma),
                out.ctypes.data_as(ctypes.c_void_p),
                0,
                0,
            )
        )
        return out

    def set_noise_model(self, nu_ht=None, nu_wie=None):
        """Coloured noise: relative coefficient variances (include/b4d.h b4d_set_noise_model); None: white."""
        if nu_ht is None:
            _check(load().b4d_set_noise_model(self._h, None, None))
            return
        a = np.ascontiguousarray(nu_ht, dtype=np.float32)
        b = np.ascontiguousarray(nu_wie, dtype=np.float32)
        _check(load().b4d_set_noise_model(self._h, a.ctypes.data_as(ctypes.c_void_p), b.ctypes.data_as(ctypes.c_void_p)))

    def stage2_matches(self, shape):
        """(widx[R, K], cnt[R]) of the last two-stage call on one volume of `shape`: window index
        (dz*Ns + dy)*Ns + dx of every match, group size per reference block."""
        R = int(load().b4d_num_refs(self._shape3(shape)))
        K = self.profile.k_wie
        widx = np.empty((R, K), dtype=np.uint16)
        cnt = np.empty((R,), dtype=np.uint8)
        _check(load().b4d_oracle_stage2_matches(self._h, widx.ctypes.data_as(ctypes.c_void_p),
                                                cnt.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(R)))
        return widx, cnt

    def accumulators(self, n):
        """(numq, wmap) int64 arrays of the last mirror filter stage (see b4d_debug_accumulators)."""
        numq = np.empty(n, dtype=np.int64)
        wmap = np.empty(n, dtype=np.int64)
        _check(load().b4d_debug_accumulators(self._h, numq.ctypes.data_as(ctypes.c_void_p),
                                             wmap.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(n)))
        return numq, wmap

    def denoise_slab(self, slab, z_begin, z_total, own_begin, own_end, sigma):
        slab = np.ascontiguousarray(slab, dtype=np.uint16)
        out = np.empty((own_end - own_begin,) + slab.shape[1:], dtype=np.float32)
        _check(
            load().b4d_denoise_slab_u16(
                self._h,
                slab.ctypes.data_as(ctypes.c_void_p),
                self._shape3(slab.shape),
                ctypes.c_int64(z_begin),
                ctypes.c_int64(z_total),
                ctypes.c_int64(own_begin),
                ctypes.c_int64(own_end),
                ctypes.c_float(sigma),
                out.ctypes.data_as(ctypes.c_void_p),
                0,
                0,
            )
        )
        return out

    def match_stage1(self, vol, sigma):
        vol = np.ascontiguousarray(vol, dtype=np.uint16)
        lib = load()
        shape = self._shape3(vol.shape)
        R = lib.b4d_num_refs(shape)
        K = self.profile.k_ht
        idx = np.empty((R, K), dtype=np.int32)
        ssd = np.empty((R, K), dtype=np.uint64)
        cnt = np.empty((R,), dtype=np.int32)
        _check(
            lib.b4d_match_stage1(
                self._h,
                vol.ctypes.data_as(ctypes.c_void_p),
                shape,
                ctypes.c_float(sigma),
                idx.ctypes.data_as(ctypes.c_void_p),
                ssd.ctypes.data_as(ctypes.c_void_p),
                cnt.ctypes.data_as(ctypes.c_void_p),
            )
        )
        return idx, ssd, cnt

    def quantize(self, x, offset_sub=0.0, offset_add=0.0, step=1.0):
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = np.empty(x.shape, dtype=np.uint16)
        _check(
            load().b4d_quantize_u16(
                self._h,
                x.ctypes.data_as(ctypes.c_void_p),
                ctypes.c_int64(x.size),
                ctypes.c_float(offset_sub),
                ctypes.c_float(offset_add),
                ctypes.c_float(step),
                out.ctypes.data_as(ctypes.c_void_p),
                0,
                0,
            )
        )
        return out


def ref_origins(n, L=4, step=3):
    """Reference-block origins along one axis (SURVEY Appendix A)."""
    o = list(range(0, n - L + 1, step))
    if (n - L) % step:
        o.append(n - L)
    return o


def match_bruteforce(vol, sigma, Ns=11, K=16, tau=2.9527):
    """Pure-NumPy instrumented matcher for tiny volumes: an independent check of
    the C++ matcher (same contract, different code)."""
    vol = np.asarray(vol).astype(np.int64)
    D, H, W = vol.shape
    r = Ns // 2
    # float32 tau and sigma, promoted to float64, exactly as the C side evaluates it
    tau_i = int(np.floor(float(np.float32(tau)) * float(np.float32(sigma)) * float(np.float32(sigma)) * 64.0))
    Hc, Wc = H - 3, W - 3
    out_idx, out_ssd, out_cnt = [], [], []
    for oz in ref_origins(D):
        for oy in ref_origins(H):
            for ox in ref_origins(W):
                ref = vol[oz : oz + 4, oy : oy + 4, ox : ox + 4]
                cand = []
                for cz in range(max(0, oz - r), min(D - 4, oz + r) + 1):
                    for cy in range(max(0, oy - r), min(H - 4, oy + r) + 1):
                        for cx in range(max(0, ox - r), min(W - 4, ox + r) + 1):
                            d = vol[cz : cz + 4, cy : cy + 4, cx : cx + 4] - ref
                            s = int((d * d).sum())
                            if s <= tau_i:
                                wi = ((cz - oz + r) * Ns + (cy - oy + r)) * Ns + (cx - ox + r)
                                cand.append((s, wi, (cz * Hc + cy) * Wc + cx))
                cand.sort()
                n = min(len(cand), K)
                kp = 1 << (n.bit_length() - 1) if n else 0
                idx = [-1] * K
                ssd = [np.iinfo(np.uint64).max] * K
                for k in range(kp):
                    idx[k] = cand[k][2]
                    ssd[k] = cand[k][0]
                out_idx.append(idx)
                out_ssd.append(ssd)
                out_cnt.append(kp)
    return (
        np.array(out_idx, dtype=np.int32),
        np.array(out_ssd, dtype=np.uint64),
        np.array(out_cnt, dtype=np.int32),
    )
