"""CPU: the oracle port against the golden vectors produced by the unmodified reference build
(tests/golden/make_golden.py), and - where the reference build is present - directly against it."""
import numpy as np
import pytest

import astc_images as I
from astc_ref import *  # noqa: F401,F403
from golden.make_golden import CASES, make_image


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_matches_golden(case, oracle, golden):
    name, gen, size, dtype, prof, bx, by, q, fl, swz = case
    img = make_image(gen, size, dtype)
    got = oracle.compress(img, prof, bx, by, q, fl, swz=list(swz))
    want = golden[name]
    assert got.shape == want.shape
    assert len(block_diff(got, want)) == 0


def test_golden_fixture_is_reproducible(reference, golden):
    """The committed fixture is what the reference build emits (guards against a stale .npz)."""
    for case in CASES[:6]:
        name, gen, size, dtype, prof, bx, by, q, fl, swz = case
        img = make_image(gen, size, dtype)
        assert same_bytes(golden[name], reference.compress(img, prof, bx, by, q, fl, swz=swz))


def test_oracle_matches_reference_on_larger_image(oracle, reference):
    img = I.photo_like(192, 160, seed=99)
    for (bx, by, q) in [(6, 6, PRE_MEDIUM), (4, 4, PRE_FAST)]:
        r = reference.compress(img, PRF_LDR, bx, by, q, FLG_SELF_DECOMPRESS_ONLY)
        o = oracle.compress(img, PRF_LDR, bx, by, q, FLG_SELF_DECOMPRESS_ONLY)
        assert same_bytes(o, r)


def test_reference_thread_invariance(reference_build):
    """The reference's output does not depend on the number of caller threads (SURVEY section 0)."""
    img = I.photo_like(96, 96, seed=5)
    a = reference_build.compress(img, PRF_LDR, 6, 6, PRE_MEDIUM, FLG_SELF_DECOMPRESS_ONLY, threads=1)
    b = reference_build.compress(img, PRF_LDR, 6, 6, PRE_MEDIUM, FLG_SELF_DECOMPRESS_ONLY, threads=4)
    assert np.array_equal(a, b)


def test_constant_block_golden_vector(oracle):
    """Known-answer: a constant LDR block is FC FD FF FF FF FF FF FF + 4 x UNORM16 (the layout the
    reference's own functional test byte-compares, Test/astc_test_functional.py:457)."""
    img = I.constant(4, 4, rgba=(255, 128, 0, 255))
    out = oracle.compress(img, PRF_LDR, 4, 4, PRE_MEDIUM, FLG_SELF_DECOMPRESS_ONLY)
    assert bytes(out[:8]) == bytes([0xFC, 0xFD, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF])
    vals = out[8:16].view(np.uint16)
    assert list(vals) == [65535, 128 * 257, 0, 65535]


@pytest.mark.parametrize("which", ["oracle", "product"])
def test_tables_equal_reference_tables_entry_by_entry(tmp_path, which):
    """tests/probe/probe_tables.cpp links the oracle's table construction with the reference's own (block modes, decimation tables
    incl. the 3D simplex ones, partitionings, coverage bitmaps, k-means texels, BISE / quantisation tables) and compares every entry:
    8 two-dimensional configurations and the ten 3D footprints. "product": the same probe over the host-side table construction of the
    CUDA library (what the kernels read), so that it is pinned to the reference directly and not through the oracle. Needs the reference
    sources: runs in the dev container only."""
    import subprocess
    src = "/root/reference/Source"
    if not os.path.isdir(src):
        pytest.skip("reference sources not here")
    exe = str(tmp_path / "probe")
    units = ["block_sizes", "partition_tables", "percentile_tables", "quantization", "weight_quant_xfer_tables", "mathlib", "mathlib_softfloat"]
    cmd = ["g++", "-std=c++14", "-O1", "-I" + src, "-DASTCENC_SSE=0", "-DASTCENC_AVX=0", "-DASTCENC_NEON=0", "-DASTCENC_POPCNT=0", "-DASTCENC_F16C=0",
           os.path.join(ROOT, "tests", "probe", "probe_tables.cpp")] + \
          ([os.path.join(ROOT, "oracle", "astc_tables.cpp")] if which == "oracle" else
           ["-DPROBE_PRODUCT=1", os.path.join(ROOT, "astc-encoder_b200", "csrc", "astc_host_tables.cpp")]) + \
          [os.path.join(src, "astcenc_%s.cpp" % u) for u in units] + ["-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "TOTAL FAILS 0" in r.stdout, r.stdout[-2000:]
    assert r.stdout.count("bsd ") == 18
