"""Image error metrics (SURVEY.md §8f rank 3): astcenc_b200_compute_error_metrics vs the oracle restatement of the
reference CLI's compute_error_metrics() (astcenccli_error_metrics.cpp:109-413).

Oracle pinning: tests/golden/golden_metrics.npz holds what the UNMODIFIED reference prints (4 decimals) for seeded image
pairs; the oracle must reproduce every printed figure. The device path reduces in parallel, so it is compared with the
oracle's raster-order double sums under a stated tolerance instead of bit for bit.
"""
import os
import numpy as np
import pytest
from astc_ref import *

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_metrics.npz")
PROD = os.path.join(ROOT, "astc-encoder_b200", "libastcenc_b200.so")

# the CLI prints %9.4f (rgb_peak: %f): half a unit of the last printed digit, plus slack for a figure sitting on a tie
PRINT_TOL = {k: 5.1e-5 for k in METRIC_FIELDS}
PRINT_TOL["rgb_peak"] = 5.1e-7

# device vs oracle: sums of ~1e3..1e7 non-negative float terms in double, different association only
LDR_RTOL = 1e-12
# HDR figures go through powf (CUDA: <= 2 ulp, glibc: <= 1 ulp) and a double acos for normals
HDR_ATOL_DB = 1e-4
ANGLE_ATOL = 1e-9


def _cases():
    g = np.load(GOLD)
    for name in g["names"]:
        name = str(name)
        hdr, normal, comps, lo, hi = [int(v) for v in g[name + "/args"]]
        yield name, g[name + "/img1"], g[name + "/img2"], dict(hdr=bool(hdr), normal=bool(normal), components=comps, fstop_lo=lo, fstop_hi=hi), g[name + "/ref"]


def _check_printed(got, ref_vec, name):
    for k, want in zip(METRIC_FIELDS, ref_vec):
        if np.isnan(want):
            continue      # figure not printed for this mode
        assert abs(got[k] - want) <= PRINT_TOL[k], (name, k, got[k], want)


def test_oracle_matches_reference_golden():
    orc = Oracle()
    n = 0
    for name, i1, i2, kw, ref in _cases():
        _check_printed(orc.error_metrics(i1, i2, **kw), ref, name)
        n += 1
    assert n >= 12


def test_oracle_matches_reference_live(reference):
    orc = Oracle()
    rng = np.random.default_rng(77)
    for trial in range(6):
        h, w = int(rng.integers(5, 60)), int(rng.integers(5, 60))
        a = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        b = np.clip(a.astype(int) + rng.integers(-20, 21, a.shape), 0, 255).astype(np.uint8)
        comps = int(rng.integers(1, 5))
        r = reference.cli_error_metrics(a, b, normal=True, components=comps)
        o = orc.error_metrics(a, b, normal=True, components=comps)
        for k, v in r.items():
            assert abs(o[k] - v) <= PRINT_TOL[k], (trial, k, o[k], v)


def test_oracle_properties():
    orc = Oracle()
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, (32, 32, 4), dtype=np.uint8)
    same = orc.error_metrics(a, a.copy())
    assert same["psnr"] == 999.0 and same["alpha_psnr"] == 999.0 and same["rgb_psnr"] == 999.0
    b = a.copy()
    b[..., 0] ^= 1      # every red value off by one: MSE = (1/255)^2 on one of 4 channels
    m = orc.error_metrics(a, b)
    d = np.float32(1.0) / np.float32(255.0)
    assert abs(m["psnr"] - 10 * np.log10(4.0 / float(d) ** 2)) < 1e-3


def _close(got, want, hdr, normal):
    for k in ("psnr", "alpha_psnr", "rgb_psnr"):
        assert got[k] == pytest.approx(want[k], rel=LDR_RTOL, abs=1e-11), k
    assert got["rgb_peak"] == want["rgb_peak"]
    for c in range(4):
        assert got["sum_squared_error"][c] == pytest.approx(want["sum_squared_error"][c], rel=LDR_RTOL), c
    if hdr:
        assert got["peak_psnr"] == pytest.approx(want["peak_psnr"], rel=LDR_RTOL, abs=1e-11)
        assert abs(got["mpsnr"] - want["mpsnr"]) <= HDR_ATOL_DB
        assert got["log_rmse"] == pytest.approx(want["log_rmse"], rel=1e-12)
    if normal:
        assert abs(got["mean_angular_error"] - want["mean_angular_error"]) <= ANGLE_ATOL
        assert abs(got["worst_angular_error"] - want["worst_angular_error"]) <= ANGLE_ATOL


@pytest.mark.gpu
def test_device_metrics_match_oracle_on_golden_pairs():
    prod = AstcencLib(PROD)
    orc = Oracle()
    for name, i1, i2, kw, ref in _cases():
        got = prod.error_metrics(i1, i2, **kw)
        _close(got, orc.error_metrics(i1, i2, **kw), kw["hdr"], kw["normal"])
        _check_printed(got, ref, name)      # and the device figures print like the reference's


@pytest.mark.gpu
def test_device_metrics_round_trip_1k():
    """compress -> decompress on the GPU, then the metrics of the pair: device vs oracle on a 1024^2 image."""
    import astc_images as I
    prod = AstcencLib(PROD)
    orc = Oracle()
    img = I.photo_like(1024, 1024, seed=9)
    blocks = prod.compress(img, PRF_LDR, 6, 6, PRE_FAST)
    dec = prod.decompress(blocks, 1024, 1024, PRF_LDR, 6, 6)
    got = prod.error_metrics(img, dec, normal=True)
    _close(got, orc.error_metrics(img, dec, normal=True), False, True)
    assert 20.0 < got["psnr"] < 80.0


@pytest.mark.gpu
def test_device_metrics_full_size_properties():
    """4096^2 (BASELINE.json's size): size-independent properties instead of the CPU oracle."""
    prod = AstcencLib(PROD)
    rng = np.random.default_rng(3)
    a = rng.integers(0, 256, (4096, 4096, 4), dtype=np.uint8)
    m = prod.error_metrics(a, a)
    assert m["psnr"] == 999.0 and m["rgb_psnr"] == 999.0 and m["alpha_psnr"] == 999.0
    b = a.copy()
    b[..., 1] ^= 1
    m = prod.error_metrics(a, b)
    d = float(np.float32(1.0) / np.float32(255.0))
    # every green value off by one: the squared error is the same float for every texel up to the rounding of
    # (g/255 - g'/255), so the sum is close to N * d^2
    assert m["sum_squared_error"][0] == 0.0 and m["sum_squared_error"][2] == 0.0 and m["sum_squared_error"][3] == 0.0
    assert m["sum_squared_error"][1] == pytest.approx(4096 * 4096 * d * d, rel=1e-6)
    assert abs(m["psnr"] - 10 * np.log10(4.0 / (d * d))) < 1e-4


@pytest.mark.gpu
def test_device_metrics_bad_params():
    prod = AstcencLib(PROD)
    a = np.zeros((8, 8, 4), dtype=np.uint8)
    with pytest.raises(RuntimeError):
        prod.error_metrics(a, a, components=0)
    with pytest.raises(RuntimeError):
        prod.error_metrics(a, a, hdr=True, fstop_lo=-200)
