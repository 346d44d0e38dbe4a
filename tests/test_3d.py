"""3D block sizes (the ten footprints 3x3x3 .. 6x6x6; /root/reference/Source/astcenc_block_sizes.cpp:1025-1190, simplex weight
infill :497-583, volume load / store astcenc_image.cpp:162-342, no mode-0 trial astcenc_compress_symbolic.cpp:1287, 3D void
extents astcenc_symbolic_physical.cpp:348-366).

CPU (-m "not gpu"): the oracle and the device source (tests/hostsim: one simulated lane, and the 32 emulated lanes of a warp)
against the unmodified reference build on seeded volumes. GPU: the CUDA library through the C ABI against the same build -
every block identical, every footprint, LDR and HDR, compression, decompression and astcenc_get_block_info."""
import ctypes as C
import os

import numpy as np
import pytest

import astc_images as I
from astc_ref import *  # noqa: F401,F403

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FOOTPRINTS = [(3, 3, 3), (4, 3, 3), (4, 4, 3), (4, 4, 4), (5, 4, 4), (5, 5, 4), (5, 5, 5), (6, 5, 5), (6, 6, 5), (6, 6, 6)]
_DT = {np.dtype(np.uint8): 0, np.dtype(np.float16): 1, np.dtype(np.float32): 2}


def ldr_volume(w, h, d, seed, kind="photo_like"):
    """(d, h, w, 4) uint8: a seeded image cut into slices (neighbouring slices are neighbouring image stripes)."""
    img = getattr(I, kind)(h * d, w, seed=seed)
    return np.ascontiguousarray(img.reshape(d, h, w, 4))


def hdr_volume(w, h, d, seed):
    return np.ascontiguousarray(I.hdr_noise(h * d, w, seed=seed).reshape(d, h, w, 4))


def _sim_compress(lib, vol, prof, fp, q, flags=0):
    d, h, w = vol.shape[:3]
    n = ((w + fp[0] - 1) // fp[0]) * ((h + fp[1] - 1) // fp[1]) * ((d + fp[2] - 1) // fp[2])
    out = np.zeros(n * 16, dtype=np.uint8)
    lib.hostsim_compress_volume.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.c_uint, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.c_uint,
                                            C.POINTER(C.c_int), C.c_void_p]
    rc = lib.hostsim_compress_volume(prof, fp[0], fp[1], fp[2], q, flags, vol.ctypes.data, _DT[vol.dtype], w, h, d, None, out.ctypes.data)
    assert rc == 0
    return out


def _sim_decompress(lib, blocks, w, h, d, prof, fp, out_type):
    out = np.zeros((d, h, w, 4), dtype=AstcencLib.NP_TYPES[out_type])
    lib.hostsim_decompress_volume.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.c_uint,
                                              C.POINTER(C.c_int)]
    rc = lib.hostsim_decompress_volume(prof, fp[0], fp[1], fp[2], 0, blocks.ctypes.data, out.ctypes.data, out_type, w, h, d, None)
    assert rc == 0
    return out


# ------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fp", FOOTPRINTS, ids=["%dx%dx%d" % f for f in FOOTPRINTS])
def test_oracle_matches_reference_build(fp, oracle, reference):
    """The oracle's restatement of the 3D tables / volume path is pinned to the unmodified reference build."""
    vol = ldr_volume(13, 11, 7, seed=fp[0] * 100 + fp[1] * 10 + fp[2])
    for q in (PRE_FASTEST, PRE_MEDIUM):
        want = reference.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q)
        got = oracle.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q)
        assert same_bytes(got, want)
    blocks = reference.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], PRE_FAST)
    assert same_bytes(oracle.decompress_volume(blocks, 13, 11, 7, PRF_LDR, fp[0], fp[1], fp[2]),
                      reference.decompress_volume(blocks, 13, 11, 7, PRF_LDR, fp[0], fp[1], fp[2]))


@pytest.mark.parametrize("fp", FOOTPRINTS, ids=["%dx%dx%d" % f for f in FOOTPRINTS])
def test_device_source_one_lane_matches_reference_build(fp, hostsim, reference):
    """The device code (state machine, arithmetic order, table layouts for 3D) compiled for the host, one simulated lane."""
    vol = ldr_volume(13, 11, 7, seed=fp[0] * 100 + fp[1] * 10 + fp[2])
    for q in (PRE_FASTEST, PRE_MEDIUM, PRE_THOROUGH):
        want = reference.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q)
        assert same_bytes(_sim_compress(hostsim, vol, PRF_LDR, fp, q), want)
    hv = hdr_volume(12, 10, 6, seed=fp[1])
    for prof in (PRF_HDR_RGB_LDR_A, PRF_HDR):
        want = reference.compress_volume(hv, prof, fp[0], fp[1], fp[2], PRE_MEDIUM)
        assert same_bytes(_sim_compress(hostsim, hv, prof, fp, PRE_MEDIUM), want)


@pytest.mark.parametrize("fp", [(3, 3, 3), (4, 4, 4), (5, 5, 4), (6, 6, 6)], ids=["3x3x3", "4x4x4", "5x5x4", "6x6x6"])
def test_device_source_32_lanes_matches_reference_build(fp, hostsim32, reference):
    """32 emulated lanes: the lane-parallel pieces at up to 216 texels (seven trips over the texels, weight lists of up to 216
    texels, the seven later simplex neighbours a moved weight invalidates in realign_weights)."""
    vol = ldr_volume(12, 10, 6, seed=31 + fp[0])
    for q in (PRE_FASTEST, PRE_MEDIUM):
        want = reference.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q)
        assert same_bytes(_sim_compress(hostsim32, vol, PRF_LDR, fp, q), want)
    v = ldr_volume(11, 9, 7, seed=5, kind="voronoi_flat")
    want = reference.compress_volume(v, PRF_LDR_SRGB, fp[0], fp[1], fp[2], PRE_MEDIUM)
    assert same_bytes(_sim_compress(hostsim32, v, PRF_LDR_SRGB, fp, PRE_MEDIUM), want)


@pytest.mark.parametrize("fp", [(3, 3, 3), (5, 4, 4), (6, 6, 6)], ids=["3x3x3", "5x4x4", "6x6x6"])
def test_device_decode_matches_reference_build(fp, hostsim, reference):
    """Decompression of real and of random blocks (error blocks, 3D void extents included), U8 and F16 output."""
    vol = ldr_volume(13, 11, 7, seed=77)
    real = reference.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], PRE_FAST)
    rnd = np.random.default_rng(fp[0]).integers(0, 256, size=real.size, dtype=np.uint8)
    # void-extent headers with assorted 3D extents (all ones = no extent, ordered, reversed = error)
    void = rnd.copy().reshape(-1, 16)
    void[:, 0] = 0xFC
    void[:, 1] = (void[:, 1] & 0xFC) | 0x01
    void[0, 1:8] = 0xFF
    void = void.reshape(-1)
    for blocks in (real, rnd, void):
        for ot in (TYPE_U8, TYPE_F16):
            want = reference.decompress_volume(blocks, 13, 11, 7, PRF_LDR, fp[0], fp[1], fp[2], out_type=ot)
            got = _sim_decompress(hostsim, blocks, 13, 11, 7, PRF_LDR, fp, ot)
            assert same_bytes(got, want)


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
def _gpu_compress(pkg, vol, prof, fp, q, flags=0):
    cfg = pkg.config_init(prof, fp[0], fp[1], q, flags, block_z=fp[2])
    ctx = pkg.Context(cfg)
    try:
        return ctx.compress_image(vol)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fp", FOOTPRINTS, ids=["%dx%dx%d" % f for f in FOOTPRINTS])
def test_cuda_volume_matches_reference_build(fp, pkg, reference):
    """astcenc_compress_image with a 3D block size: every block of a 96 x 80 x 24 volume identical to the reference build
    (ragged edges in all three axes), -fastest / -medium / -thorough; HDR profiles on F16 data."""
    vol = ldr_volume(97, 83, 25, seed=fp[0] * 100 + fp[1] * 10 + fp[2])
    for q in (PRE_FASTEST, PRE_MEDIUM, PRE_THOROUGH):
        if q == PRE_THOROUGH:
            vol = vol[:13, :40, :50]
        want = reference.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q)
        got = _gpu_compress(pkg, vol, PRF_LDR, fp, q)
        assert same_bytes(got, want), "%s q=%s: the %d blocks differ from the reference build's" % (fp, q, len(got) // 16)
    hv = hdr_volume(41, 37, 13, seed=fp[1])
    for prof in (PRF_HDR_RGB_LDR_A, PRF_HDR):
        want = reference.compress_volume(hv, prof, fp[0], fp[1], fp[2], PRE_MEDIUM)
        assert same_bytes(_gpu_compress(pkg, hv, prof, fp, PRE_MEDIUM), want)


@pytest.mark.gpu
def test_cuda_volume_content_classes(pkg, reference):
    """Partition-search stress, noise, alpha masks, flat volumes (constant blocks), one slice only (dim_z < block_z)."""
    for fp in ((4, 4, 4), (6, 6, 6)):
        for kind in ("voronoi_flat", "uniform_noise", "alpha_mask", "smooth_gradient"):
            v = ldr_volume(50, 46, 14, seed=9, kind=kind)
            want = reference.compress_volume(v, PRF_LDR_SRGB, fp[0], fp[1], fp[2], PRE_MEDIUM)
            assert same_bytes(_gpu_compress(pkg, v, PRF_LDR_SRGB, fp, PRE_MEDIUM), want), (fp, kind)
        flat = np.ascontiguousarray(np.broadcast_to(np.array([12, 200, 99, 255], dtype=np.uint8), (9, 20, 22, 4)))
        assert same_bytes(_gpu_compress(pkg, flat, PRF_LDR, fp, PRE_MEDIUM), reference.compress_volume(flat, PRF_LDR, fp[0], fp[1], fp[2], PRE_MEDIUM))
        one = ldr_volume(33, 29, 1, seed=4)
        assert same_bytes(_gpu_compress(pkg, one, PRF_LDR, fp, PRE_MEDIUM), reference.compress_volume(one, PRF_LDR, fp[0], fp[1], fp[2], PRE_MEDIUM))


@pytest.mark.gpu
@pytest.mark.parametrize("fp", [(3, 3, 3), (5, 4, 4), (6, 6, 6)], ids=["3x3x3", "5x4x4", "6x6x6"])
def test_cuda_volume_decode_and_block_info(fp, pkg, reference):
    """astcenc_decompress_image and astcenc_get_block_info with a 3D block size, against the reference build."""
    vol = ldr_volume(45, 39, 17, seed=77)
    real = reference.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], PRE_FAST)
    rnd = np.random.default_rng(fp[0]).integers(0, 256, size=real.size, dtype=np.uint8)
    cfg = pkg.config_init(PRF_LDR, fp[0], fp[1], PRE_MEDIUM, 0, block_z=fp[2])
    ctx = pkg.Context(cfg)
    try:
        for blocks in (real, rnd):
            for dt, ot in ((np.uint8, TYPE_U8), (np.float16, TYPE_F16)):
                want = reference.decompress_volume(blocks, 45, 39, 17, PRF_LDR, fp[0], fp[1], fp[2], out_type=ot)
                got = ctx.decompress_image(blocks, 45, 39, dtype=dt, dim_z=17)
                assert same_bytes(got, want)
        err = np.abs(ctx.decompress_image(real, 45, 39, dim_z=17).astype(np.int32) - vol.astype(np.int32))
        assert err.mean() < 30.0      # it really is the volume (6x6x6 is 0.59 bits per texel and the slices are image stripes)
    finally:
        ctx.close()
    prod = AstcencLib(os.path.join(ROOT, "astc-encoder_b200", "libastcenc_b200.so"))
    some = np.concatenate([real[:40 * 16], rnd[:40 * 16]])
    assert same_bytes(prod.block_infos(some, PRF_LDR, fp[0], fp[1], bz=fp[2]), reference.block_infos(some, PRF_LDR, fp[0], fp[1], bz=fp[2]))
