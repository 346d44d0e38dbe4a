"""Decompression (SURVEY.md section 8f, first "next" row): astcenc_decompress_image.

Fixtures: tests/golden/golden_decode.npz, written by the unmodified reference build (tests/golden/make_golden_decode.py).
CPU: the oracle restatement and the host simulation of the device source must reproduce them byte for byte.
GPU: the CUDA path, through the C ABI, must reproduce them too; plus the reference's API error order."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
from astc_ref import *  # noqa: E402,F401,F403
from make_golden_decode import DCASES, make_blocks  # noqa: E402

NP = {TYPE_U8: np.uint8, TYPE_F16: np.float16, TYPE_F32: np.float32}


@pytest.fixture(scope="module")
def golden_decode():
    return np.load(os.path.join(HERE, "golden", "golden_decode.npz"))


def _case_blocks(i, golden):
    name, source, size, prof, bx, by, ot, fl, swz = DCASES[i]
    return make_blocks(source, size, bx, by, golden, 100 + i)


@pytest.mark.parametrize("i", range(len(DCASES)), ids=[c[0] for c in DCASES])
def test_oracle_decode_matches_reference_fixture(i, oracle, golden, golden_decode):
    name, source, size, prof, bx, by, ot, fl, swz = DCASES[i]
    img = oracle.decompress(_case_blocks(i, golden), size[1], size[0], prof, bx, by, ot, fl, list(swz))
    assert np.array_equal(np.ascontiguousarray(img).view(np.uint8).reshape(-1), golden_decode[name])


@pytest.mark.parametrize("i", range(len(DCASES)), ids=[c[0] for c in DCASES])
def test_device_source_host_simulation_decode(i, hostsim, golden, golden_decode):
    name, source, size, prof, bx, by, ot, fl, swz = DCASES[i]
    blocks = np.ascontiguousarray(_case_blocks(i, golden), dtype=np.uint8)
    out = np.zeros((size[0], size[1], 4), dtype=NP[ot])
    sw = (C.c_int * 4)(*swz)
    assert hostsim.hostsim_decompress_image(prof, bx, by, fl, blocks.ctypes.data, out.ctypes.data, ot, size[1], size[0], sw) == 0
    assert np.array_equal(out.view(np.uint8).reshape(-1), golden_decode[name])


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(DCASES)), ids=[c[0] for c in DCASES])
def test_cuda_decode_matches_reference_fixture(i, pkg, golden, golden_decode):
    name, source, size, prof, bx, by, ot, fl, swz = DCASES[i]
    cfg = pkg.config_init(prof, bx, by, PRE_MEDIUM, fl)
    ctx = pkg.Context(cfg)
    try:
        img = ctx.decompress_image(_case_blocks(i, golden), size[1], size[0], dtype=NP[ot], swizzle=swz)
        assert ctx.launch_count() >= 1
    finally:
        ctx.close()
    assert np.array_equal(np.ascontiguousarray(img).view(np.uint8).reshape(-1), golden_decode[name])


@pytest.mark.gpu
def test_cuda_round_trip_and_random_blocks_against_oracle(pkg, oracle):
    """compress -> decompress on the GPU equals the oracle's decode of the same blocks; so do 4096 random blocks."""
    import astc_images as I
    img = I.photo_like(120, 132, seed=21)
    cfg = pkg.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, 0)
    ctx = pkg.Context(cfg)
    try:
        blocks = ctx.compress_image(img)
        got = ctx.decompress_image(blocks, 132, 120)
        want = oracle.decompress(blocks, 132, 120, PRF_LDR, 6, 6, TYPE_U8)
        assert np.array_equal(got, want)
        err = np.abs(got.astype(np.int32) - img.astype(np.int32))
        assert err.mean() < 6.0        # it really is the image
        rb = np.random.default_rng(5).integers(0, 256, size=4096 * 16, dtype=np.uint8)
        got = ctx.decompress_image(rb, 64 * 6, 64 * 6, dtype=np.float16)
        want = oracle.decompress(rb, 64 * 6, 64 * 6, PRF_LDR, 6, 6, TYPE_F16)
        assert np.array_equal(got.view(np.uint16), want.view(np.uint16))
    finally:
        ctx.close()


@pytest.mark.gpu
def test_decompress_error_order_and_slices(pkg, oracle):
    """Check order of astcenc_decompress_image (astcenc_entry.cpp:1285-1330) and a 3-slice volume of 2D blocks."""
    cfg = pkg.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, 0)
    ctx = pkg.Context(cfg)
    try:
        blocks = np.zeros(4 * 16, dtype=np.uint8)
        with pytest.raises(pkg.AstcencError) as e:
            ctx.decompress_image(blocks, 12, 12, thread_index=1)
        assert e.value.code == pkg.ERR_BAD_PARAM
        with pytest.raises(pkg.AstcencError) as e:
            ctx.decompress_image(blocks, 12, 12, swizzle=(0, 1, 2, 7))
        assert e.value.code == pkg.ERR_BAD_SWIZZLE
        with pytest.raises(pkg.AstcencError) as e:
            ctx.decompress_image(blocks[:48], 12, 12)
        assert e.value.code == pkg.ERR_OUT_OF_MEM
        rb = np.random.default_rng(9).integers(0, 256, size=3 * 9 * 16, dtype=np.uint8)
        vol = ctx.decompress_image(rb, 18, 18, dim_z=3)
        for z in range(3):
            want = oracle.decompress(rb[z * 9 * 16:(z + 1) * 9 * 16], 18, 18, PRF_LDR, 6, 6, TYPE_U8)
            assert np.array_equal(vol[z], want)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_get_block_info_matches_reference(pkg, reference, golden):
    """astcenc_get_block_info: every field of the struct equals the reference build's, on real, random and void-extent blocks."""
    prod = AstcencLib(os.path.join(ROOT, "astc-encoder_b200", "libastcenc_b200.so"))
    rng = np.random.default_rng(31)
    streams = [(golden["photo_6x6_medium"][:64 * 16], PRF_LDR, 6, 6), (golden["voronoi_8x8_thorough"][:48 * 16], PRF_LDR, 8, 8),
               (golden["hdr_f16_6x6_medium"][:48 * 16], PRF_HDR, 6, 6), (rng.integers(0, 256, size=96 * 16, dtype=np.uint8), PRF_LDR, 5, 5),
               (make_blocks("void", (24, 24), 6, 6, golden, 3), PRF_HDR, 6, 6)]
    for blocks, prof, bx, by in streams:
        want = reference.block_infos(blocks, prof, bx, by)
        got = prod.block_infos(blocks, prof, bx, by)
        assert same_bytes(got, want)
