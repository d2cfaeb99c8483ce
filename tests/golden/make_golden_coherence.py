"""Golden vectors for the spatial-coherence gate, made by RUNNING THE REFERENCE.

    python tests/golden/make_golden_coherence.py REFERENCE_CHECKOUT

Imports machine_learning/metrics.py straight from REFERENCE_CHECKOUT/src (read-only, nothing copied) and records, for
seeded patches (labels uint64, raw float32 counts): patch_has_incoherent_segment(labels, raw, ...)
(metrics.py:189-260) and, per segment, local_autocorr(raw, labels == id, lag) (:64-112) and
highfreq_energy_fraction(raw, labels == id, smooth = gaussian_filter(raw, sigma)) (:115-155).  Cases, in the spirit
of tests/test_metrics.py:24-40: a smooth PSF-like blob (coherent), a salt-and-pepper block (the artifact), both in
one patch, a thin faint neurite, a segment below the voxel minimum, a constant segment (degenerate variance), a
ragged shape, other lags / sigmas / thresholds.  The inputs are not stored (the seeded noise does not compress): the
tests rebuild them with cases() and check them against the SHA-256 digest kept in tests/golden/reference_coherence.npz
next to the reference's outputs.
"""
import hashlib
import importlib.util
import os
import sys

import numpy as np
from scipy import ndimage

REF_SUBDIR = os.path.join("src", "aind_exaspim_image_compression", "machine_learning")
HERE = os.path.dirname(os.path.abspath(__file__))


def _load(ref, name):
    spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(ref, REF_SUBDIR, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def smooth_blob(shape, lo, hi, amp, sigma):
    v = np.zeros(shape, dtype=np.float32)
    v[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = amp
    return ndimage.gaussian_filter(v, sigma)


def salt_pepper(shape, lo, hi, amp, rate, rng):
    v = np.zeros(shape, dtype=np.float32)
    region = np.zeros(shape, dtype=bool)
    region[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = True
    v[(rng.random(shape) < rate) & region] = amp
    return v, region


def digest(labels, raw):
    """SHA-256 of one case's inputs (shape, uint64 labels, float32 raw) as 32 uint8."""
    h = hashlib.sha256(repr(labels.shape).encode())
    h.update(np.ascontiguousarray(labels, np.uint64).tobytes())
    h.update(np.ascontiguousarray(raw, np.float32).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def cases():
    rng = np.random.default_rng(20261020)
    out = []
    shape = (48, 48, 48)
    noise = lambda s: rng.normal(0.0, 12.0, s).astype(np.float32)  # noqa: E731
    # 1. coherent blob only
    blob = smooth_blob(shape, (8, 8, 8), (40, 40, 40), 800.0, 2.0)
    lab = np.zeros(shape, np.uint64)
    lab[blob > 50] = 7
    out.append((lab, blob + noise(shape), {}))
    # 2. salt-and-pepper artifact only
    sp, region = salt_pepper(shape, (8, 8, 8), (40, 40, 40), 900.0, 0.4, rng)
    lab = np.zeros(shape, np.uint64)
    lab[region] = 123456789012345
    out.append((lab, sp + noise(shape), {}))
    # 3. both in one patch, plus a tiny segment below the voxel minimum and a constant one
    blob = smooth_blob(shape, (4, 4, 4), (20, 44, 44), 700.0, 2.0)
    sp, region = salt_pepper(shape, (28, 6, 6), (44, 40, 40), 900.0, 0.35, rng)
    raw = blob + sp + noise(shape)
    lab = np.zeros(shape, np.uint64)
    lab[blob > 60] = 3
    lab[region] = 2 ** 40 + 5
    lab[22:24, 2:5, 2:5] = 9          # 18 voxels: ignored
    raw[24:27, 44:48, 44:48] = 500.0   # constant segment: degenerate variance, autocorr unmeasurable
    lab[24:27, 44:48, 44:48] = 11
    out.append((lab, raw, {}))
    # 4. thin faint but smooth neurite: low autocorrelation from thinness, low high-frequency energy
    v = np.zeros(shape, np.float32)
    v[24, 10:40, 24] = 600.0
    thin = ndimage.gaussian_filter(v, 1.2)
    lab = np.zeros(shape, np.uint64)
    lab[thin > 8] = 42
    out.append((lab, thin + 0.2 * noise(shape), {}))
    # 5. ragged shape, two artifacts with different rates, other parameters
    shape2 = (21, 34, 29)
    sp1, r1 = salt_pepper(shape2, (2, 2, 2), (10, 30, 27), 1200.0, 0.5, rng)
    sp2, r2 = salt_pepper(shape2, (12, 4, 3), (20, 20, 25), 400.0, 0.15, rng)
    lab = np.zeros(shape2, np.uint64)
    lab[r1] = 1
    lab[r2] = 2
    raw = sp1 + sp2 + noise(shape2)
    out.append((lab, raw, dict(coherence_lag=1, smooth_sigma=1.5)))
    out.append((lab, raw, dict(min_autocorr=0.05, max_highfreq_frac=0.9)))
    out.append((lab, raw, dict(coherence_lag=3, smooth_sigma=0.7, min_segment_voxels=5000)))
    # 6. no labels at all
    out.append((np.zeros(shape2, np.uint64), raw, {}))
    return out


def main(ref):
    me = _load(ref, "metrics")
    data = {}
    cs = cases()
    for i, (lab, raw, kw) in enumerate(cs):
        verdict = bool(me.patch_has_incoherent_segment(lab, raw, **kw))
        lag, sig = kw.get("coherence_lag", 2), kw.get("smooth_sigma", 1.0)
        smooth = ndimage.gaussian_filter(np.asarray(raw, dtype=np.float64), sigma=sig)
        ids = np.unique(lab[lab > 0])
        sc = np.array([[float((lab == l).sum()), me.local_autocorr(raw, lab == l, lag=lag),
                        me.highfreq_energy_fraction(raw, lab == l, smooth=smooth)] for l in ids], dtype=np.float64).reshape(-1, 3)
        data["digest%d" % i] = digest(lab, raw)
        data["ids%d" % i] = ids.astype(np.uint64)
        data["scores%d" % i] = sc
        data["verdict%d" % i] = np.array(verdict)
        data["params%d" % i] = np.array([kw.get("min_autocorr", 0.4), kw.get("max_highfreq_frac", 0.35),
                                        kw.get("min_segment_voxels", 50), sig, lag], dtype=np.float64)
        print("case %d shape %s segments %d verdict %s" % (i, lab.shape, len(ids), verdict), sc.round(4).tolist())
    data["n"] = np.array(len(cs))
    np.savez_compressed(os.path.join(HERE, "reference_coherence.npz"), **data)


if __name__ == "__main__":
    main(sys.argv[1])
