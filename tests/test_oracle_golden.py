"""The oracle against golden vectors produced by RUNNING the reference
(tests/golden/make_golden.py imports /root/reference's transforms.py and
metrics.py).  Pins every step around BM4D that exists in the reference tree.
BM4D itself is PARITY UNPINNED (closed wheel bm4d==4.2.5, absent)."""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def test_quantize_matches_reference_offset_transform(gold, oracle_lib):
    x = gold["quant_x"]
    for i, off in enumerate(gold["quant_offsets"]):
        want = gold["quant_q%d" % i]
        got = oracle_lib.quantize_reference(x, offset_add=float(off))
        assert got.dtype == np.uint16 and np.array_equal(got, want)
        # the K7 contract at step = 1, offset_sub = 0 degenerates to the reference bit for bit
        assert np.array_equal(oracle_lib.quantize_noise_scaled(x, 0.0, float(off), 1.0), want)
        # and so does the C restatement
        o = oracle_lib.Oracle("f64")
        assert np.array_equal(o.quantize(x, 0.0, float(off), 1.0), want)


def test_quantize_matches_reference_asinh_inverse(gold, oracle_lib):
    assert np.array_equal(oracle_lib.quantize_reference(gold["asinh_counts"]), gold["asinh_q"])


def test_estimate_offset_matches_reference(gold, oracle_lib):
    from b4d.sharding import stats_from_hist

    data, pos = gold["offset_data"], 0
    for n, p, want in zip(gold["offset_n"], gold["offset_pct"], gold["offset_val"]):
        s = data[pos : pos + n]
        pos += n
        assert oracle_lib.estimate_offset(s, percentile=float(p)) == want
        # host-side statistic from the exact histogram (what ranks all-gather)
        st = stats_from_hist(np.bincount(s, minlength=65536), float(p))
        assert st["offset"] == want, (n, p, st["offset"], want)


def test_mad_sigma_matches_reference_mask(gold, oracle_lib):
    from b4d.sharding import stats_from_hist

    for k in range(4):
        raw = gold["mask_raw%d" % k]
        med, mad, sigma = oracle_lib.robust_sigma(raw)
        st = stats_from_hist(np.bincount(raw.reshape(-1), minlength=65536))
        assert (st["median"], st["mad"], st["sigma"]) == (med, mad, sigma)
        for kk in (3, 6):
            want = np.unpackbits(gold["mask_m%d_k%d" % (k, kk)])[: raw.size].astype(bool).reshape(raw.shape)
            # metrics.py:58 in float32
            thr = np.float32(med) + np.float32(kk) * np.float32(sigma)
            got = raw.astype(np.float32) > thr
            assert np.array_equal(got, want)


def _mask_cases():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_masks.npz"))
    for i in range(int(g["count"][0])):
        ci, off, k, dil = g["par%d" % i]
        u = g["u%d" % int(ci)]
        want = np.unpackbits(g["m%d" % i])[: u.size].astype(bool).reshape(u.shape)
        yield u, float(off), float(k), int(dil), want


def test_foreground_mask_restatements_match_the_reference(oracle_lib):
    """make_foreground_mask (metrics.py:32-61) run live by tests/golden/make_golden_masks.py on
    raw = uint16 - offset: the NumPy restatement (shift-based dilation) and the C++ one behind the
    oracle's C ABI (selection medians, 6-neighbour passes) both reproduce its masks exactly."""
    import ctypes

    lib = oracle_lib.load()
    n = 0
    for u, off, k, dil, want in _mask_cases():
        raw = oracle_lib.read_counts(u, np.float32(off))
        assert np.array_equal(oracle_lib.make_foreground_mask_reference(raw, k, dil), want)
        out = np.empty(u.shape, np.uint8)
        offs = np.array([off], np.float32)
        rc = lib.b4d_foreground_mask_u16(None, ctypes.c_void_p(u.ctypes.data), ctypes.c_int64(1),
                                         (ctypes.c_int64 * 3)(*u.shape), ctypes.c_void_p(offs.ctypes.data),
                                         ctypes.c_float(k), ctypes.c_int(dil), ctypes.c_void_p(out.ctypes.data), 0, 0)
        assert rc == 0 and np.array_equal(out.astype(bool), want)
        n += 1
    assert n == 45


def test_truncating_variant(oracle_lib):
    x = np.array([-3.2, 0.0, 0.9, 1.5, 2.5, 65535.9], dtype=np.float32)
    assert oracle_lib.quantize_truncating(x).tolist() == [0, 0, 0, 1, 2, 65535]


def _coherence_cases():
    """The reference's outputs with their inputs, rebuilt from the seeded recipe of
    tests/golden/make_golden_coherence.py and checked byte for byte against the digests stored with the outputs."""
    from golden import make_golden_coherence

    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_coherence.npz"))
    inputs = make_golden_coherence.cases()
    assert len(inputs) == int(g["n"])
    for i, (lab, raw, _) in enumerate(inputs):
        assert np.array_equal(make_golden_coherence.digest(lab, raw), g["digest%d" % i]), \
            "case %d: the rebuilt inputs are not the ones the reference was run on" % i
        p = g["params%d" % i]
        kw = dict(min_autocorr=float(p[0]), max_highfreq_frac=float(p[1]), min_segment_voxels=int(p[2]),
                  smooth_sigma=float(p[3]), coherence_lag=int(p[4]))
        yield lab, raw, kw, g["ids%d" % i], g["scores%d" % i], bool(g["verdict%d" % i])


def test_coherence_gate_restatement_matches_the_reference(oracle_lib):
    """np_oracle's restatement of the sampler's coherence gate against outputs of the LIVE reference
    (tests/golden/make_golden_coherence.py: patch_has_incoherent_segment, local_autocorr,
    highfreq_energy_fraction of metrics.py): verdicts equal, per-segment scores equal to 1e-12."""
    n = 0
    for lab, raw, kw, ids, scores, verdict in _coherence_cases():
        sc = oracle_lib.coherence_scores_reference(lab, raw, kw["smooth_sigma"], kw["coherence_lag"])
        assert sorted(sc) == [int(v) for v in ids]
        for lid, want in zip(ids, scores):
            got = sc[int(lid)]
            assert got[0] == int(want[0])
            assert abs(got[1] - want[1]) <= 1e-12 and abs(got[2] - want[2]) <= 1e-12
        assert oracle_lib.patch_has_incoherent_segment_reference(lab, raw, **kw) == verdict
        n += 1
    assert n >= 8
