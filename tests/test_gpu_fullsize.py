"""GPU: whole-image equality with the unmodified reference build at BASELINE.json's full sizes (configs[0..3]), and the
host-pointer / sharding paths added in round 2 (banded uploads, stream ordering of one context, the sharded and batch
entry points with a world of one). Bit-exact on the 16-byte blocks; everything goes through the C ABI."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import astc_images as I
from astc_ref import *  # noqa: F401,F403

pytestmark = pytest.mark.gpu
S = FLG_SELF_DECOMPRESS_ONLY
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gpu(pkg):
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return pkg


# (name, generator, size, profile, block, quality): BASELINE.json configs[0..3] at their full sizes
FULL = [
    ("config0_512_4x4_fast", "photo_like", 512, PRF_LDR, 4, PRE_FAST),
    ("config1_4096_6x6_medium", "photo_like", 4096, PRF_LDR, 6, PRE_MEDIUM),
    ("config2_4096_8x8_thorough", "photo_like", 4096, PRF_LDR, 8, PRE_THOROUGH),
    ("config3_2048_hdr_6x6_medium", "hdr_noise", 2048, PRF_HDR, 6, PRE_MEDIUM),
]


@pytest.mark.parametrize("case", FULL, ids=[c[0] for c in FULL])
def test_whole_image_equals_reference_build(case, gpu, reference):
    """Every block of the full-size workload image, product vs the reference library (its output recorded as a digest)."""
    name, gen, dim, prof, b, q = case
    img = getattr(I, gen)(dim, dim, seed=2024)
    cfg = gpu.config_init(prof, b, b, q, S)
    ctx = gpu.Context(cfg)
    try:
        got = ctx.compress_image(img)
    finally:
        ctx.close()
    want = reference.compress(img, prof, b, b, q, S)
    assert same_bytes(got, want), "the %d blocks differ from the reference build's" % (len(got) // 16)


def test_banded_upload_equals_single_copy(gpu):
    """astcenc_compress_image uploads the image in bands under the wave-0 set-up (ASTCENC_B200_UPLOAD_BANDS, read when the
    context is made): any band count gives the same bytes, for even and ragged heights."""
    outs = {}
    for bands in ("1", "4", "8"):
        os.environ["ASTCENC_B200_UPLOAD_BANDS"] = bands
        try:
            cfg = gpu.config_init(PRF_LDR, 6, 6, PRE_FAST, S)
            ctx = gpu.Context(cfg)
            for (h, w) in ((768, 512), (1001, 333), (40, 64)):
                img = I.photo_like(h, w, seed=h)
                outs.setdefault((h, w), []).append(ctx.compress_image(img))
            ctx.close()
        finally:
            del os.environ["ASTCENC_B200_UPLOAD_BANDS"]
    for k, v in outs.items():
        assert all(np.array_equal(v[0], x) for x in v[1:]), k


def test_sub_slab_pipelines_equal_the_plain_wave_loop(gpu):
    """A pass may run as P independent sub-slab pipelines on P streams (ASTCENC_B200_PIPES, read when the context is made):
    every P gives the bytes of the plain wave loop, host-pointer path and device-resident path alike, ragged sizes included."""
    import torch
    dev = torch.device("cuda", 0)
    img = I.photo_like(1500, 1210, seed=12)
    d_img = torch.from_numpy(img).to(dev)
    outs = []
    for pipes in ("1", "2", "4", "8"):
        os.environ["ASTCENC_B200_PIPES"] = pipes
        try:
            ctx = gpu.Context(gpu.config_init(PRF_LDR, 5, 5, PRE_FAST, S))
            host = ctx.compress_image(img).copy()
            nbx, nby = ctx.blocks(1210, 1500)
            d_out = torch.zeros(nbx * nby * 16, dtype=torch.uint8, device=dev)
            st = torch.cuda.Stream(device=dev)
            torch.cuda.synchronize()
            for _ in range(2):
                ctx.compress_device(d_img.data_ptr(), gpu.TYPE_U8, 1210, 1500, d_out.data_ptr(), stream=st.cuda_stream)
            torch.cuda.synchronize()
            assert np.array_equal(d_out.cpu().numpy(), host)
            # a slab of the image through the same machinery
            r0, r1 = 31, 257
            d_slab = torch.zeros((r1 - r0) * nbx * 16, dtype=torch.uint8, device=dev)
            ctx.compress_device(d_img.data_ptr(), gpu.TYPE_U8, 1210, 1500, d_slab.data_ptr(), block_row0=r0, block_rows=r1 - r0, stream=st.cuda_stream)
            torch.cuda.synchronize()
            assert np.array_equal(d_slab.cpu().numpy(), host[r0 * nbx * 16:r1 * nbx * 16])
            outs.append(host)
            ctx.close()
        finally:
            del os.environ["ASTCENC_B200_PIPES"]
    assert all(np.array_equal(outs[0], o) for o in outs[1:])


def test_one_context_two_streams_are_ordered(gpu):
    """Two device-resident passes of ONE context on different streams share the context's scratch: the library orders
    them (mutex + event chain), so both results are right whatever the streams do."""
    import torch
    dev = torch.device("cuda", 0)
    cfg = gpu.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, S)
    ctx = gpu.Context(cfg)
    ref_ctx = gpu.Context(cfg)
    try:
        imgs = [I.photo_like(600, 600, seed=s) for s in (1, 2, 3, 4)]
        want = [ref_ctx.compress_image(im) for im in imgs]
        d_imgs = [torch.from_numpy(im).to(dev) for im in imgs]
        nbx, nby = ctx.blocks(600, 600)
        d_outs = [torch.zeros(nbx * nby * 16, dtype=torch.uint8, device=dev) for _ in imgs]
        streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
        torch.cuda.synchronize()
        for rep in range(3):
            for i, (di, do) in enumerate(zip(d_imgs, d_outs)):
                ctx.compress_device(di.data_ptr(), gpu.TYPE_U8, 600, 600, do.data_ptr(), stream=streams[i & 1].cuda_stream)
            # and the host-pointer path on the context's own stream in between
            mid = ctx.compress_image(imgs[0])
            assert np.array_equal(mid, want[0])
        torch.cuda.synchronize()
        for do, w in zip(d_outs, want):
            assert np.array_equal(do.cpu().numpy(), w)
    finally:
        ctx.close()
        ref_ctx.close()


def test_entry_points_restore_the_current_device(gpu):
    import torch
    before = torch.cuda.current_device()
    cfg = gpu.config_init(PRF_LDR, 4, 4, PRE_FAST, S)
    ctx = gpu.Context(cfg)
    ctx.compress_image(I.photo_like(32, 32, seed=1))
    ctx.close()
    assert torch.cuda.current_device() == before


def test_sharded_and_batch_entry_points_world_of_one(gpu):
    """With one rank the collective entry points run locally (no NCCL communicator) and return the bytes of
    astcenc_compress_image: slab mode on one image, batch mode over several images with overlapped uploads."""
    cfg = gpu.config_init(PRF_LDR, 6, 6, PRE_MEDIUM, S)
    ctx = gpu.Context(cfg)
    try:
        ctx.comm_init(0, 1)
        imgs = [I.photo_like(300, 420, seed=s) for s in range(5)]
        want = [ctx.compress_image(im).copy() for im in imgs]
        got = ctx.compress_image_sharded(imgs[2])
        assert np.array_equal(got, want[2])
        outs = [np.zeros_like(w) for w in want]
        ctx.compress_batch(imgs, outs)
        for o, w in zip(outs, want):
            assert np.array_equal(o, w)
        # slab arithmetic of the C ABI equals the Python helper
        for world in (1, 2, 3, 8):
            for r in range(world):
                a, n = ctx.slab_rows(300, r, world)
                r0, r1 = gpu.slab_rows((300 + 5) // 6, r, world)
                assert (a, n) == (r0, r1 - r0)
        # errors: mixed sizes in a batch, bad root
        with pytest.raises(gpu.AstcencError):
            ctx.compress_batch([imgs[0], I.photo_like(64, 64, seed=1)], [outs[0], outs[1]])
        with pytest.raises(gpu.AstcencError):
            ctx.compress_image_sharded(imgs[0], root=3)
    finally:
        ctx.close()


def test_two_ranks_nccl_slab_and_batch(gpu, tmp_path):
    """Two GPUs (skipped on a one-GPU box): slab mode and batch mode through NCCL are byte-identical to one GPU."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = os.path.join(ROOT, "tests", "multi_gpu_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29613", script, str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert os.path.exists(os.path.join(str(tmp_path), "ok"))
