"""GPU: the CUDA path (through the astcenc.h C ABI of libastcenc_b200.so) against the golden vectors of the
reference, the oracle port, the reference build's recorded outputs (tests/golden/golden_reference.npz), and - at
BASELINE.json's full sizes - through size-independent properties (block independence, slab invariance,
determinism). Bit-exact: every comparison is on the 16-byte physical blocks."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

import astc_images as I
from astc_ref import *  # noqa: F401,F403
from golden.make_golden import CASES, make_image

pytestmark = pytest.mark.gpu
S = FLG_SELF_DECOMPRESS_ONLY


@pytest.fixture(scope="module")
def gpu(pkg):
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return pkg


def gpu_compress(pkg, img, prof, bx, by, q, fl=0, swz=(0, 1, 2, 3), threads=1, **ov):
    cfg = pkg.config_init(prof, bx, by, q, fl, **ov)
    ctx = pkg.Context(cfg, thread_count=threads)
    try:
        out = ctx.compress_image(img, swizzle=swz)
        assert ctx.launch_count() >= 1        # the CUDA kernel really ran
        return out
    finally:
        ctx.close()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_cuda_matches_golden(case, gpu, golden):
    name, gen, size, dtype, prof, bx, by, q, fl, swz = case
    img = make_image(gen, size, dtype)
    got = gpu_compress(gpu, img, prof, bx, by, q, fl, swz)
    assert len(block_diff(got, golden[name])) == 0


@pytest.mark.parametrize("cfgcase", [
    (PRF_LDR, 6, 6, PRE_MEDIUM, S), (PRF_LDR, 4, 4, PRE_FAST, S), (PRF_LDR, 8, 8, PRE_THOROUGH, S),
    (PRF_LDR, 5, 5, PRE_MEDIUM, S | FLG_USE_DECODE_UNORM8), (PRF_LDR_SRGB, 10, 10, PRE_MEDIUM, S),
    (PRF_LDR, 12, 12, PRE_MEDIUM, S), (PRF_LDR, 6, 6, PRE_VERYTHOROUGH, S), (PRF_LDR, 8, 6, 75.0, S),
])
def test_cuda_matches_oracle_on_seeded_images(cfgcase, gpu, oracle):
    prof, bx, by, q, fl = cfgcase
    for gen, size in [("photo_like", (192, 160)), ("uniform_noise", (72, 72)), ("smooth_gradient", (96, 96)),
                      ("voronoi_flat", (90, 90)), ("alpha_mask", (101, 77))]:
        if q >= PRE_VERYTHOROUGH:
            size = (min(size[0], 48), min(size[1], 48))
        img = getattr(I, gen)(*size, seed=77)
        want = oracle.compress(img, prof, bx, by, q, fl)
        got = gpu_compress(gpu, img, prof, bx, by, q, fl)
        d = block_diff(got, want)
        assert len(d) == 0, (gen, len(d), d[:5])


def test_cuda_matches_reference_build(gpu, reference):
    """Same binary interface, same inputs: the product library and the unmodified reference library."""
    img = I.photo_like(512, 512, seed=5)
    for (bx, by, q) in [(4, 4, PRE_FAST), (6, 6, PRE_MEDIUM)]:
        want = reference.compress(img, PRF_LDR, bx, by, q, S)
        got = gpu_compress(gpu, img, PRF_LDR, bx, by, q, S)
        assert same_bytes(got, want)


def test_hdr_matches_oracle(gpu, oracle):
    img = I.hdr_noise(126, 126, seed=9)
    for prof in (PRF_HDR, PRF_HDR_RGB_LDR_A):
        want = oracle.compress(img, prof, 6, 6, PRE_MEDIUM, S)
        got = gpu_compress(gpu, img, prof, 6, 6, PRE_MEDIUM, S)
        assert len(block_diff(got, want)) == 0


def test_tuning_overrides_follow_the_oracle(gpu, oracle):
    """Power-user overrides change the search tree the same way (1 partition only / 2-plane disabled gate of SURVEY 7.2)."""
    img = I.photo_like(96, 96, seed=21)
    want = oracle.compress(img, PRF_LDR, 6, 6, PRE_MEDIUM, S, partition_count_limit=1, plane2_correlation=0.0)
    got = gpu_compress(gpu, img, PRF_LDR, 6, 6, PRE_MEDIUM, S, tune_partition_count_limit=1, tune_2plane_early_out_limit_correlation=0.0)
    assert len(block_diff(got, want)) == 0


# ---- full-size properties (BASELINE.json configs) -------------------------------------------------

@pytest.fixture(scope="module")
def image_4k():
    return I.photo_like(4096, 4096, seed=2024)


def test_4k_6x6_medium_block_sample_against_oracle(gpu, oracle, image_4k):
    """Blocks are independent: a mosaic of randomly sampled 6x6 blocks must compress to exactly the blocks the
    full 4096^2 run produced at those positions."""
    bx = by = 6
    got = gpu_compress(gpu, image_4k, PRF_LDR, bx, by, PRE_MEDIUM, S).reshape(-1, 16)
    blocks_x = (4096 + bx - 1) // bx
    rng = np.random.default_rng(1)
    n = 1024
    xs = rng.integers(0, 4096 // bx, n)
    ys = rng.integers(0, 4096 // by, n)
    mosaic = np.zeros((32 * by, 32 * bx, 4), np.uint8)
    for i, (x, y) in enumerate(zip(xs, ys)):
        mosaic[(i // 32) * by:(i // 32 + 1) * by, (i % 32) * bx:(i % 32 + 1) * bx] = image_4k[y * by:(y + 1) * by, x * bx:(x + 1) * bx]
    want = oracle.compress(mosaic, PRF_LDR, bx, by, PRE_MEDIUM, S).reshape(-1, 16)
    sel = got[ys * blocks_x + xs]
    assert np.array_equal(sel, want)


def test_4k_slab_sharding_is_invisible(gpu, image_4k):
    """Block-row slabs (the multi-GPU partitioning) concatenate to exactly the single-launch output, and the
    result is deterministic run to run."""
    import torch
    pkg = gpu
    cfg = pkg.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, S)
    ctx = pkg.Context(cfg)
    whole = ctx.compress_image(image_4k)
    again = ctx.compress_image(image_4k)
    assert np.array_equal(whole, again)
    d_img = torch.from_numpy(image_4k).cuda()
    nbx, nby = ctx.blocks(4096, 4096)
    d_out = torch.zeros(nbx * nby * 16, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for world in (2, 3, 8):
        d_out.zero_()
        for r in range(world):
            r0, r1 = pkg.slab_rows(nby, r, world)
            ctx.compress_device(d_img.data_ptr(), TYPE_U8, 4096, 4096, d_out.data_ptr() + r0 * nbx * 16, r0, r1 - r0, stream=stream)
        torch.cuda.synchronize()
        assert np.array_equal(d_out.cpu().numpy(), whole), world
    ctx.close()


def test_4k_8x8_thorough_block_sample(gpu, oracle, image_4k):
    bx = by = 8
    crop = image_4k[:1024, :1024]
    got = gpu_compress(gpu, crop, PRF_LDR, bx, by, PRE_THOROUGH, S).reshape(-1, 16)
    rng = np.random.default_rng(2)
    n = 256
    xs = rng.integers(0, 1024 // bx, n)
    ys = rng.integers(0, 1024 // by, n)
    mosaic = np.zeros((16 * by, 16 * bx, 4), np.uint8)
    for i, (x, y) in enumerate(zip(xs, ys)):
        mosaic[(i // 16) * by:(i // 16 + 1) * by, (i % 16) * bx:(i % 16 + 1) * bx] = crop[y * by:(y + 1) * by, x * bx:(x + 1) * bx]
    want = oracle.compress(mosaic, PRF_LDR, bx, by, PRE_THOROUGH, S).reshape(-1, 16)
    assert np.array_equal(got[ys * (1024 // bx) + xs], want)


# ---- API behaviour (mirrors Source/UnitTest/test_encode.cpp) ----------------------------------------

def _ctx(pkg, threads=1, **kw):
    cfg = pkg.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, S, **kw)
    return pkg.Context(cfg, thread_count=threads)


def test_error_order_matches_reference(gpu):
    pkg = gpu
    lib = pkg.lib()
    ctx = _ctx(pkg)
    img = np.zeros((8, 8, 4), np.uint8)
    slices = (C.c_void_p * 1)(img.ctypes.data)
    image = pkg.Image(8, 8, 1, TYPE_U8, slices)
    out = np.zeros(64, np.uint8)
    good = pkg.Swizzle(0, 1, 2, 3)
    assert lib.astcenc_compress_image(ctx.handle, C.byref(image), C.byref(pkg.Swizzle(0, 1, 2, 6)), out.ctypes.data, out.nbytes, 0) == 7   # BAD_SWIZZLE (Z invalid)
    assert lib.astcenc_compress_image(ctx.handle, C.byref(image), C.byref(good), out.ctypes.data, out.nbytes, 1) == 3                      # thread_index >= count
    assert lib.astcenc_compress_image(ctx.handle, C.byref(pkg.Image(0, 8, 1, TYPE_U8, slices)), C.byref(good), out.ctypes.data, out.nbytes, 0) == 3
    assert lib.astcenc_compress_image(ctx.handle, C.byref(image), C.byref(good), out.ctypes.data, 63, 0) == 1                               # short buffer: OUT_OF_MEM
    huge = pkg.Image(0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, TYPE_U8, slices)
    assert lib.astcenc_compress_image(ctx.handle, C.byref(huge), C.byref(good), out.ctypes.data, out.nbytes, 0) == 3                        # size overflow: BAD_PARAM
    assert lib.astcenc_compress_image(ctx.handle, C.byref(image), C.byref(good), out.ctypes.data, out.nbytes, 0) == 0
    ctx.close()
    dcfg = pkg.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, FLG_DECOMPRESS_ONLY)
    dctx = pkg.Context(dcfg)
    assert lib.astcenc_compress_image(dctx.handle, C.byref(image), C.byref(good), out.ctypes.data, out.nbytes, 0) == 9                      # BAD_CONTEXT
    assert lib.astcenc_compress_reset(dctx.handle) == 9
    dctx.close()


def test_multiple_caller_threads(gpu, oracle):
    """thread_count callers may enter compress_image; any subset does; all return SUCCESS with the full image done."""
    pkg = gpu
    img = I.photo_like(120, 120, seed=4)
    want = oracle.compress(img, PRF_LDR, 6, 6, PRE_MEDIUM, S)
    ctx = _ctx(pkg, threads=4)
    for callers in (4, 2):
        out = np.zeros(len(want), np.uint8)
        slices = (C.c_void_p * 1)(img.ctypes.data)
        image = pkg.Image(120, 120, 1, TYPE_U8, slices)
        sw = pkg.Swizzle(0, 1, 2, 3)
        errs = [None] * callers

        def run(i):
            errs[i] = pkg.lib().astcenc_compress_image(ctx.handle, C.byref(image), C.byref(sw), out.ctypes.data, out.nbytes, i)
        ts = [threading.Thread(target=run, args=(i,)) for i in range(callers)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert errs == [0] * callers
        assert np.array_equal(out, want)
        assert pkg.lib().astcenc_compress_reset(ctx.handle) == 0
    ctx.close()


def test_child_context_shares_tables(gpu, oracle):
    pkg = gpu
    img = I.photo_like(60, 60, seed=8)
    want = oracle.compress(img, PRF_LDR, 6, 6, PRE_MEDIUM, S)
    parent = _ctx(pkg)
    child = C.c_void_p()
    assert pkg.lib().astcenc_context_alloc(None, 1, C.byref(child), parent.handle) == 0
    out = np.zeros(len(want), np.uint8)
    slices = (C.c_void_p * 1)(img.ctypes.data)
    image = pkg.Image(60, 60, 1, TYPE_U8, slices)
    sw = pkg.Swizzle(0, 1, 2, 3)
    assert pkg.lib().astcenc_compress_image(child, C.byref(image), C.byref(sw), out.ctypes.data, out.nbytes, 0) == 0
    assert np.array_equal(out, want)
    pkg.lib().astcenc_context_free(child)
    parent.close()


def test_nan_inf_inputs_do_not_crash_and_match(gpu, oracle):
    """test_encode.cpp:170-299: +-Inf / NaN texels in F32 input for LDR, HDR and HDR_RGB_LDR_A."""
    rng = np.random.default_rng(3)
    img = rng.uniform(-1, 2, size=(24, 24, 4)).astype(np.float32)
    img[3, 3, 0] = np.nan
    img[9, 2, 1] = np.inf
    img[13, 20, 3] = -np.inf
    for prof in (PRF_LDR, PRF_HDR, PRF_HDR_RGB_LDR_A):
        want = oracle.compress(img, prof, 6, 6, PRE_MEDIUM, S)
        got = gpu_compress(gpu, img, prof, 6, 6, PRE_MEDIUM, S)
        assert len(block_diff(got, want)) == 0


def test_volume_of_2d_slices(gpu, oracle):
    """dim_z > 1 with 2D blocks = independent slices laid out one after another."""
    vol = np.stack([I.photo_like(36, 42, seed=s) for s in (1, 2, 3)])
    cfg = gpu.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, S)
    ctx = gpu.Context(cfg)
    got = ctx.compress_image(vol)
    ctx.close()
    want = np.concatenate([oracle.compress(vol[z], PRF_LDR, 6, 6, PRE_MEDIUM, S) for z in range(3)])
    assert np.array_equal(got, want)


@pytest.mark.parametrize("driver", ["lockstep", "warp"])
def test_single_kernel_drivers_agree(gpu, oracle, monkeypatch, driver):
    """The single-kernel drivers kept for A/B measurements (ASTCENC_B200_DRIVER) produce the same bytes as the wave pipeline."""
    monkeypatch.setenv("ASTCENC_B200_DRIVER", driver)
    img = I.photo_like(96, 96, seed=12)
    want = oracle.compress(img, PRF_LDR, 6, 6, PRE_MEDIUM, S)
    got = gpu_compress(gpu, img, PRF_LDR, 6, 6, PRE_MEDIUM, S)
    assert np.array_equal(got, want)


def test_batched_slabs_and_stage_barriers(gpu, oracle, monkeypatch):
    """Small record batches (several pipeline passes per image) and the optional stage barriers change nothing."""
    img = I.photo_like(192, 160, seed=13)
    want = oracle.compress(img, PRF_LDR, 6, 6, PRE_MEDIUM, S)
    monkeypatch.setenv("ASTCENC_B200_BATCH_BLOCKS", "100")
    assert np.array_equal(gpu_compress(gpu, img, PRF_LDR, 6, 6, PRE_MEDIUM, S), want)
    monkeypatch.setenv("ASTCENC_B200_SYNC_MASK", "0xFF")
    assert np.array_equal(gpu_compress(gpu, img, PRF_LDR, 6, 6, PRE_MEDIUM, S), want)


@pytest.mark.parametrize("env", [{"ASTCENC_B200_STAGE_REFINE": "1"}, {"ASTCENC_B200_STAGE_SETUP": "0"}, {"ASTCENC_B200_STAGE_SETUP": "1"}])
def test_table_staging_changes_nothing(gpu, oracle, monkeypatch, env):
    """Decimation / colour tables read from shared memory or from global memory: same bytes."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    for img, prof, bx, by, q in ((I.photo_like(120, 96, seed=21), PRF_LDR, 6, 6, PRE_MEDIUM), (I.voronoi_flat(64, 64, seed=3), PRF_LDR, 8, 8, PRE_MEDIUM),
                                 (I.hdr_noise(48, 48, seed=2), PRF_HDR, 5, 4, PRE_MEDIUM)):
        want = oracle.compress(img, prof, bx, by, q, S)
        assert np.array_equal(gpu_compress(gpu, img, prof, bx, by, q, S), want)


def test_mode0_disabled_and_partition_limits(gpu, oracle):
    """Presets without the mode-0 trial (thorough and up) and with 1..4 partitions take the unshared set-up path."""
    img = I.voronoi_flat(96, 96, seed=5)
    for q in (PRE_THOROUGH, PRE_FASTEST):
        want = oracle.compress(img, PRF_LDR, 5, 5, q, S)
        assert np.array_equal(gpu_compress(gpu, img, PRF_LDR, 5, 5, q, S), want)
