"""Records tests/golden/golden_reference.npz: what the UNMODIFIED reference build (oracle/_ref, built by oracle/Makefile where the
reference's sources are present) returns for every call the tests make through the `reference` fixture (astc_ref.RecordedReference).

The calls below repeat the tests' own, with the same seeded inputs; a call a test makes that is not recorded here fails that
test with a KeyError. Run from the repository root:  python tests/golden/make_golden_reference.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS)
sys.path.insert(0, HERE)
import astc_images as I  # noqa: E402
from astc_ref import *  # noqa: E402,F401,F403
from make_golden import CASES, make_image  # noqa: E402
from make_golden_decode import make_blocks  # noqa: E402
from test_3d import FOOTPRINTS, hdr_volume, ldr_volume  # noqa: E402
from test_gpu_fullsize import FULL  # noqa: E402
from test_host_logic import BLOCKS, PRESET_POINTS  # noqa: E402

S = FLG_SELF_DECOMPRESS_ONLY
THREADS = max(1, len(os.sched_getaffinity(0)))


def volumes_3d(ref):
    """tests/test_3d.py"""
    for fp in FOOTPRINTS:
        vol = ldr_volume(13, 11, 7, seed=fp[0] * 100 + fp[1] * 10 + fp[2])
        for q in (PRE_FASTEST, PRE_MEDIUM, PRE_THOROUGH):
            ref.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q)
        blocks = ref.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], PRE_FAST)
        ref.pin()
        ref.decompress_volume(blocks, 13, 11, 7, PRF_LDR, fp[0], fp[1], fp[2])
        hv = hdr_volume(12, 10, 6, seed=fp[1])
        for prof in (PRF_HDR_RGB_LDR_A, PRF_HDR):
            ref.compress_volume(hv, prof, fp[0], fp[1], fp[2], PRE_MEDIUM)
    for fp in [(3, 3, 3), (4, 4, 4), (5, 5, 4), (6, 6, 6)]:
        vol = ldr_volume(12, 10, 6, seed=31 + fp[0])
        for q in (PRE_FASTEST, PRE_MEDIUM):
            ref.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q)
        ref.compress_volume(ldr_volume(11, 9, 7, seed=5, kind="voronoi_flat"), PRF_LDR_SRGB, fp[0], fp[1], fp[2], PRE_MEDIUM)
    for fp in [(3, 3, 3), (5, 4, 4), (6, 6, 6)]:
        real = ref.compress_volume(ldr_volume(13, 11, 7, seed=77), PRF_LDR, fp[0], fp[1], fp[2], PRE_FAST)
        ref.pin()
        rnd = np.random.default_rng(fp[0]).integers(0, 256, size=real.size, dtype=np.uint8)
        void = rnd.copy().reshape(-1, 16)
        void[:, 0] = 0xFC
        void[:, 1] = (void[:, 1] & 0xFC) | 0x01
        void[0, 1:8] = 0xFF
        for blocks in (real, rnd, void.reshape(-1)):
            for ot in (TYPE_U8, TYPE_F16):
                ref.decompress_volume(blocks, 13, 11, 7, PRF_LDR, fp[0], fp[1], fp[2], out_type=ot)
    # GPU tests
    for fp in FOOTPRINTS:
        vol = ldr_volume(97, 83, 25, seed=fp[0] * 100 + fp[1] * 10 + fp[2])
        for q in (PRE_FASTEST, PRE_MEDIUM, PRE_THOROUGH):
            if q == PRE_THOROUGH:
                vol = vol[:13, :40, :50]
            ref.compress_volume(vol, PRF_LDR, fp[0], fp[1], fp[2], q, threads=THREADS)
        hv = hdr_volume(41, 37, 13, seed=fp[1])
        for prof in (PRF_HDR_RGB_LDR_A, PRF_HDR):
            ref.compress_volume(hv, prof, fp[0], fp[1], fp[2], PRE_MEDIUM, threads=THREADS)
    for fp in ((4, 4, 4), (6, 6, 6)):
        for kind in ("voronoi_flat", "uniform_noise", "alpha_mask", "smooth_gradient"):
            ref.compress_volume(ldr_volume(50, 46, 14, seed=9, kind=kind), PRF_LDR_SRGB, fp[0], fp[1], fp[2], PRE_MEDIUM, threads=THREADS)
        flat = np.ascontiguousarray(np.broadcast_to(np.array([12, 200, 99, 255], dtype=np.uint8), (9, 20, 22, 4)))
        ref.compress_volume(flat, PRF_LDR, fp[0], fp[1], fp[2], PRE_MEDIUM)
        ref.compress_volume(ldr_volume(33, 29, 1, seed=4), PRF_LDR, fp[0], fp[1], fp[2], PRE_MEDIUM)
    for fp in [(3, 3, 3), (5, 4, 4), (6, 6, 6)]:
        real = ref.compress_volume(ldr_volume(45, 39, 17, seed=77), PRF_LDR, fp[0], fp[1], fp[2], PRE_FAST, threads=THREADS)
        ref.pin()
        rnd = np.random.default_rng(fp[0]).integers(0, 256, size=real.size, dtype=np.uint8)
        for blocks in (real, rnd):
            for ot in (TYPE_U8, TYPE_F16):
                ref.decompress_volume(blocks, 45, 39, 17, PRF_LDR, fp[0], fp[1], fp[2], out_type=ot)
        ref.block_infos(np.concatenate([real[:40 * 16], rnd[:40 * 16]]), PRF_LDR, fp[0], fp[1], bz=fp[2])


def configs(ref):
    """tests/test_host_logic.py"""
    for profile in (PRF_LDR_SRGB, PRF_LDR, PRF_HDR_RGB_LDR_A, PRF_HDR):
        for (bx, by) in BLOCKS:
            for q in PRESET_POINTS:
                for fl in (0, FLG_MAP_NORMAL, FLG_MAP_RGBM, FLG_USE_PERCEPTUAL | FLG_SELF_DECOMPRESS_ONLY):
                    ref.config(profile, bx, by, q, fl)


def images_2d(ref):
    """tests/test_oracle_golden.py, test_gpu_parity.py, test_decode.py, test_gpu_fullsize.py"""
    for case in CASES[:6]:
        name, gen, size, dtype, prof, bx, by, q, fl, swz = case
        ref.compress(make_image(gen, size, dtype), prof, bx, by, q, fl, swz=swz)
    img = I.photo_like(192, 160, seed=99)
    for (bx, by, q) in [(6, 6, PRE_MEDIUM), (4, 4, PRE_FAST)]:
        ref.compress(img, PRF_LDR, bx, by, q, S)
    img = I.photo_like(512, 512, seed=5)
    for (bx, by, q) in [(4, 4, PRE_FAST), (6, 6, PRE_MEDIUM)]:
        ref.compress(img, PRF_LDR, bx, by, q, S, threads=THREADS)
    golden = np.load(os.path.join(HERE, "golden_blocks.npz"))
    rng = np.random.default_rng(31)
    streams = [(golden["photo_6x6_medium"][:64 * 16], PRF_LDR, 6, 6), (golden["voronoi_8x8_thorough"][:48 * 16], PRF_LDR, 8, 8),
               (golden["hdr_f16_6x6_medium"][:48 * 16], PRF_HDR, 6, 6), (rng.integers(0, 256, size=96 * 16, dtype=np.uint8), PRF_LDR, 5, 5),
               (make_blocks("void", (24, 24), 6, 6, golden, 3), PRF_HDR, 6, 6)]
    for blocks, prof, bx, by in streams:
        ref.block_infos(blocks, prof, bx, by)
    for name, gen, dim, prof, b, q in FULL:
        print("  full size:", name, flush=True)
        ref.compress(getattr(I, gen)(dim, dim, seed=2024), prof, b, b, q, S, threads=THREADS)


def metrics(ref):
    """tests/test_metrics.py"""
    rng = np.random.default_rng(77)
    for trial in range(6):
        h, w = int(rng.integers(5, 60)), int(rng.integers(5, 60))
        a = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        b = np.clip(a.astype(int) + rng.integers(-20, 21, a.shape), 0, 255).astype(np.uint8)
        comps = int(rng.integers(1, 5))
        ref.cli_error_metrics(a, b, normal=True, components=comps)


def main():
    assert have_ref() and have_ref_metrics(), "build the reference first: make -C oracle ref"
    ref = RecordedReference(live=ref_lib())
    for part in (volumes_3d, configs, images_2d, metrics):
        print(part.__name__, flush=True)
        part(ref)
    kept, digests = ref.save()
    print("%s: %d outputs whole, %d as digests, %d bytes" % (REF_RECORD, kept, digests, os.path.getsize(REF_RECORD)))


if __name__ == "__main__":
    main()
