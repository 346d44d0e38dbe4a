#!/usr/bin/env python
"""bench.py - Mtexels/s of the ASTC compress hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C] [--mode M]     the CUDA path
  python bench.py --impl reference [--config C] ...                               the reference's own CPU implementation (oracle/_ref)

--config  0  512x512 LDR RGBA8, 4x4, -fast          (BASELINE.json configs[0], the reference's CPU-runnable case)
          1  4096x4096 LDR RGBA8, 6x6, -medium      (configs[1], the headline; default)
          2  4096x4096 LDR RGBA8, 8x8, -thorough    (configs[2])
          3  2048x2048 HDR RGBA F16, 6x6, -medium, HDR profile (-cH)   (configs[3])
          4  batch of 8 x N images of config 1      (configs[4]: 64 x 4096^2 over 8 GPUs)

A "step" = one pass of the block compressor over the config's image (per GPU). Synthetic, seeded images (tests/astc_images.py).

value : whole-job Mtexels/s with the image already resident in HBM: CUDA events on the launching stream around the
        pipeline pass (N > 1: one image per rank + the payload gather to rank 0), L2 flushed between steps.
e2e   : the same metric through the C ABI with plain (pageable) HOST buffers - what the reference's callers pass -
        H2D of the image and D2H of the blocks inside the timed region.
          N = 1: astcenc_compress_image()
          N > 1: astcenc_b200_compress_batch() - every rank uploads / searches its own images (upload of image i+1 under
                 the search of image i), payloads gathered to rank 0 over NCCL inside the library
slab  : (N > 1, extra object) ONE image cut into block-row slabs over the N ranks through astcenc_b200_compress_image_sharded():
        strong scaling of a single image, with the gather's own device time.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

PRF_LDR, PRF_HDR = 1, 3
FLAGS = 32               # ASTCENC_FLG_SELF_DECOMPRESS_ONLY, what the reference CLI sets for -cl / -cH
CONFIGS = {
    0: dict(dim=512, block=4, quality=10.0, preset="fast", profile=PRF_LDR, pname="LDR", dtype="u8", tag="configs[0]"),
    1: dict(dim=4096, block=6, quality=60.0, preset="medium", profile=PRF_LDR, pname="LDR", dtype="u8", tag="configs[1]"),
    2: dict(dim=4096, block=8, quality=98.0, preset="thorough", profile=PRF_LDR, pname="LDR", dtype="u8", tag="configs[2]"),
    3: dict(dim=2048, block=6, quality=60.0, preset="medium", profile=PRF_HDR, pname="HDR", dtype="f16", tag="configs[3]"),
    4: dict(dim=4096, block=6, quality=60.0, preset="medium", profile=PRF_LDR, pname="LDR", dtype="u8", tag="configs[4]"),
}
IMAGES_PER_GPU = 8       # configs[4]: 64 images over 8 GPUs


def workload_name(c):
    cfg = CONFIGS[c]
    kind = "LDR RGBA8" if cfg["dtype"] == "u8" else "HDR RGBA F16"
    s = "%dx%d %s, %dx%d block, -%s" % (cfg["dim"], cfg["dim"], kind, cfg["block"], cfg["block"], cfg["preset"])
    if cfg["profile"] == PRF_HDR:
        s += ", HDR profile"
    return s + " (BASELINE.json %s)" % cfg["tag"]


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def host_info():
    """What the CPU arm can really use: affinity mask, cgroup CPU quota, CPU model (os.cpu_count() alone lies in containers)."""
    info = {"cpu_count": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["cpu_count"]
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                        quota = q / float(f2.read().split()[0])
            break
        except Exception:
            continue
    info["cgroup_quota_cores"] = quota
    model = None
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    info["cpu_model"] = model
    usable = info["affinity"]
    if quota is not None:
        usable = max(1, min(usable, int(math.ceil(quota))))
    info["usable_cores"] = usable
    return info


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            p = [x.strip() for x in l.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def make_image(c, seed):
    import astc_images
    cfg = CONFIGS[c]
    # (C-contiguous: the device-resident path uploads the array's memory as it lies; the generators may return other strides)
    if cfg["dtype"] == "f16":
        return np.ascontiguousarray(astc_images.hdr_noise(cfg["dim"], cfg["dim"], seed=seed, dtype=np.float16))
    return np.ascontiguousarray(astc_images.photo_like(cfg["dim"], cfg["dim"], seed=seed))


def variant(image, k):
    """Image k of a batch: the base image shifted / mirrored (distinct blocks, same statistics, no 6 s generator run per image)."""
    if k == 0:
        return image
    out = np.roll(image, (37 * k, 91 * k), axis=(0, 1))
    if k & 1:
        out = out[:, ::-1]
    return np.ascontiguousarray(out)


class ReferenceRunner:
    """The unmodified reference build (oracle/_ref) on the host cores. The context (block-size tables, ~0.1 s) is made
    once, outside every timed region - the metric is compression throughput, as for the GPU arm."""

    def __init__(self, c, threads):
        import astc_ref
        import ctypes as C
        self.cfg = CONFIGS[c]
        self.threads = threads
        self.lib = astc_ref.ref_lib()
        rcfg = self.lib.config(self.cfg["profile"], self.cfg["block"], self.cfg["block"], self.cfg["quality"], FLAGS)
        self.ctx = C.c_void_p()
        err = self.lib.lib.astcenc_context_alloc(C.byref(rcfg), threads, C.byref(self.ctx), None)
        assert err == 0, err

    def run(self, image, repeats=1):
        """best seconds per image over `repeats` runs; the blocks of the last run are kept in self.last"""
        best = 1e30
        for _ in range(repeats):
            t0 = time.perf_counter()
            self.last = self.lib.compress_ctx(self.ctx, image, self.cfg["block"], self.cfg["block"], threads=self.threads)
            best = min(best, time.perf_counter() - t0)
        return best

    def close(self):
        if self.ctx:
            self.lib.lib.astcenc_context_free(self.ctx)
            self.ctx = None


def cpu_baseline(c, image, max_seconds=20.0):
    import astc_ref
    cfg = CONFIGS[c]
    hi = host_info()
    texels = image.shape[0] * image.shape[1]
    if not astc_ref.have_ref():
        # fall back to the oracle port (single thread) on a crop
        crop = np.ascontiguousarray(image[:512, :512])
        o = astc_ref.Oracle()
        t0 = time.perf_counter()
        o.compress(crop, cfg["profile"], cfg["block"], cfg["block"], cfg["quality"], FLAGS)
        dt = time.perf_counter() - t0
        return {"value": crop.shape[0] * crop.shape[1] / dt / 1e6, "unit": "Mtexels/s", "cores": 1, "kind": "port", "sample": "512x512 crop of the workload image, 1 thread", "host": hi}
    threads = hi["usable_cores"]
    runner = ReferenceRunner(c, threads)
    t = runner.run(image, 1)
    reps = int(max(1, min(4, max_seconds / max(t, 1e-3) - 1)))
    t = min(t, runner.run(image, reps))
    runner.close()
    return {"value": texels / t / 1e6, "unit": "Mtexels/s", "cores": threads, "kind": "reference", "host": hi,
            "sample": "whole workload image, best of %d, %d caller threads (= usable cores: affinity %d, cgroup quota %s), astcenc avx2 invariance build"
                      % (reps + 1, threads, hi["affinity"], hi["cgroup_quota_cores"])}


DUMP_LIMIT = 63 << 20     # the dump stays under 64 MiB, .npy headers included


def dump_outputs(path, outputs):
    """Write each payload as <path>/<name>.npy: one row of 16 float32 byte values per block. Payloads over DUMP_LIMIT in
    all are cut to the same fixed, seeded sample of block rows, whose indices go to <name>_rows.npy."""
    os.makedirs(path, exist_ok=True)
    n = sum(a.size for a in outputs.values()) // 16
    # a row takes 64 bytes, and 8 more for its index once the rows are sampled
    frac = 1.0 if n * 64 <= DUMP_LIMIT else DUMP_LIMIT / (n * 72)
    for name, blocks in outputs.items():
        rows = np.asarray(blocks, dtype=np.uint8).reshape(-1, 16)
        if frac < 1.0:
            keep = int(len(rows) * frac)
            idx = np.sort(np.random.default_rng(0).choice(len(rows), size=keep, replace=False))
            rows = rows[idx]
            np.save(os.path.join(path, name + "_rows.npy"), idx.astype(np.float64))
        np.save(os.path.join(path, name + ".npy"), rows.astype(np.float32))


def traffic_from_profile():
    """DRAM bytes of one pipeline pass (all stage-kernel launches of one image), summed from the committed ncu capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get("dram_bytes_per_pass")
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS))
    ap.add_argument("--mode", default="auto", choices=["auto", "batch", "slab", "replica"],
                    help="N > 1: which library path the e2e figure uses (auto = batch, and the slab numbers as an extra object)")
    ap.add_argument("--images-per-gpu", type=int, default=0, help="batch mode: images per rank and step (default 8: BASELINE.json configs[4] is 64 images over 8 GPUs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the blocks the last timed step produced (N > 1: every rank's payload as gathered on rank 0) to DIR/*.npy, "
                                                           "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    c = args.config
    cfg = CONFIGS[c]
    DIM, BLOCK = cfg["dim"], cfg["block"]
    W = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 0)
    K = args.steps
    metric = "Mtexels/s at 4K RGBA 6x6 -medium" if c in (1, 4) else "Mtexels/s at %s" % workload_name(c).split(" (")[0]
    config = {"workload": workload_name(c), "block": "%dx%d" % (BLOCK, BLOCK), "preset": cfg["preset"], "profile": cfg["pname"],
              "l2": "flushed between timed steps (256 MiB memset)"}

    if args.impl == "reference":
        # rank 0 alone times the reference's CPU implementation; other ranks exit without work
        if rank != 0:
            return
        image = make_image(c, 2024)
        hi = host_info()
        threads = hi["usable_cores"]
        runner = ReferenceRunner(c, threads)
        for _ in range(min(W, 2)):
            runner.run(image)
        t0 = time.perf_counter()
        for _ in range(K):
            runner.run(image)
        dt = (time.perf_counter() - t0) / K
        runner.close()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"blocks": runner.last})
        v = DIM * DIM / dt / 1e6
        line = {"impl": "reference", "metric": metric, "value": v, "unit": "Mtexels/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "images_per_step": 1,
                "cpu_baseline": {"value": v, "unit": "Mtexels/s", "cores": threads, "kind": "reference", "host": hi,
                                 "sample": "whole workload image per step, %d caller threads (= usable cores: affinity %d, cgroup quota %s), astcenc avx2 invariance build"
                                           % (threads, hi["affinity"], hi["cgroup_quota_cores"])},
                "e2e": {"value": v, "unit": "Mtexels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    pkg = g.load_package()
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    base = make_image(c, 2024)                             # the workload image (the reference arm compresses the same one)
    image = variant(base, rank)                            # every rank has its own image of the batch
    acfg = pkg.config_init(cfg["profile"], BLOCK, BLOCK, cfg["quality"], FLAGS)
    ctx = pkg.Context(acfg)
    nbx, nby = ctx.blocks(DIM, DIM)
    payload = nbx * nby * 16
    bpt = image.dtype.itemsize * 4
    image_bytes = DIM * DIM * bpt
    algo_bytes = image_bytes + payload                     # read every texel once, write 16 B per block (SURVEY 8d)
    dtype_id = pkg.TYPE_U8 if cfg["dtype"] == "u8" else pkg.TYPE_F16
    d_img = torch.from_numpy(image.view(np.uint8) if image.dtype != np.uint8 else image).to(dev)
    d_out = torch.empty(payload, dtype=torch.uint8, device=dev)
    gather_list = [torch.empty(payload, dtype=torch.uint8, device=dev) for _ in range(world)] if (world > 1 and rank == 0) else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # a non-default stream: the C ABI treats stream 0 as "use the context's own stream", and CUDA events must be
    # recorded on the stream the kernel is launched on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    def step(timed_events=None):
        flush.zero_()
        if timed_events is not None:
            timed_events[0].record(stream)
        ctx.compress_device(d_img.data_ptr(), dtype_id, DIM, DIM, d_out.data_ptr(), stream=stream.cuda_stream)
        if world > 1:
            dist.gather(d_out, gather_list, dst=0)
        if timed_events is not None:
            timed_events[1].record(stream)

    for _ in range(W):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(K):
        step(evs[k])
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    launches = ctx.launch_count() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs) / K
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # copied before the passes below overwrite d_out
        if world > 1:
            outputs = {"blocks_rank%d" % r: buf.cpu().numpy() for r, buf in enumerate(gather_list)}
        else:
            outputs = {"blocks": d_out.cpu().numpy()}
        dump_outputs(args.dump_outputs, outputs)

    # kernel-only duration (roofline): events tightly around the kernel on its stream, no gather
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(K, 5))]
    for a, b in kev:
        flush.zero_()
        a.record(stream)
        ctx.compress_device(d_img.data_ptr(), dtype_id, DIM, DIM, d_out.data_ptr(), stream=stream.cuda_stream)
        b.record(stream)
    torch.cuda.synchronize()
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / len(kev)
    # one more pass with an event after every launch: how the pass splits over the four stage kernels
    ctx.stage_timing(True)
    flush.zero_()
    ctx.compress_device(d_img.data_ptr(), dtype_id, DIM, DIM, d_out.data_ptr(), stream=stream.cuda_stream)
    torch.cuda.synchronize()
    stage_ms, stage_launches = ctx.stage_timing(False, fetch=True)
    dev_blocks = d_out.cpu().numpy()

    # ---- end to end through the C ABI with plain host buffers (H2D + search + D2H inside the timed region) ----
    e2e_steps = min(K, 5)
    slab = None
    e2e_mode = "astcenc_compress_image, pageable host buffers"
    images_e2e = 1
    if world == 1 and c != 4:
        h_out = np.empty(payload, dtype=np.uint8)
        for _ in range(2):
            ctx.compress_image(image, out=h_out)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for _ in range(e2e_steps):
            ctx.compress_image(image, out=h_out)
        e2e_s = (time.perf_counter() - t1) / e2e_steps
        assert np.array_equal(h_out, dev_blocks), "host-pointer path and device-resident path disagree"
        e2e_h2d, e2e_d2h = image_bytes, payload
    else:
        uid = None
        if world > 1:
            box = [pkg.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            uid = box[0]
        ctx.comm_init(rank, world, uid)
        mode = args.mode if args.mode != "auto" else "batch"
        per_gpu = args.images_per_gpu or IMAGES_PER_GPU
        if mode in ("batch", "replica"):
            # image i of the batch lives on rank i % world; rank r holds images r, r + world, ...
            n_img = per_gpu * world
            mine = {i: variant(base, i) for i in range(rank, n_img, world)}
            images = [mine.get(i) for i in range(n_img)]
            outs = [np.empty(payload, dtype=np.uint8) for _ in range(n_img)] if rank == 0 else None
            ctx.compress_batch(images, outs)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            batch_steps = min(K, 3)
            t1 = time.perf_counter()
            for _ in range(batch_steps):
                ctx.compress_batch(images, outs)
            e2e_s = (time.perf_counter() - t1) / batch_steps
            images_e2e = n_img
            e2e_mode = "astcenc_b200_compress_batch: %d images per rank and step, image i on rank i %% %d, upload of the next image under the search of the current one, payloads to rank 0 over NCCL (library), pageable host buffers" % (per_gpu, world)
            if rank == 0:
                # image `rank`'s payload must equal what the device-resident path produced for the same image
                assert np.array_equal(outs[0], dev_blocks), "batch path and device-resident path disagree"
            e2e_h2d, e2e_d2h = image_bytes * n_img, payload * n_img
        else:
            e2e_s = None
        # slab mode: ONE image (the base image) over all ranks
        h_full = np.empty(payload, dtype=np.uint8) if rank == 0 else None
        for _ in range(2):
            ctx.compress_image_sharded(base, out=h_full)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        slab_steps = min(K, 5)
        cms, gms = [], []
        t1 = time.perf_counter()
        for _ in range(slab_steps):
            ctx.compress_image_sharded(base, out=h_full)
            a_ms, g_ms = ctx.comm_last_timing()
            cms.append(a_ms)
            gms.append(g_ms)
        slab_s = (time.perf_counter() - t1) / slab_steps
        st = torch.tensor([slab_s * 1e3, float(np.mean(cms)), float(np.mean(gms))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(st, op=dist.ReduceOp.MAX)
        slab_ms, slab_search_ms, slab_gather_ms = [float(x) for x in st.cpu()]
        if rank == 0:
            if world > 1 or c != 4:
                ref_ctx = pkg.Context(acfg)
                want = ref_ctx.compress_image(base)
                ref_ctx.close()
                assert np.array_equal(h_full, want), "slab-sharded payload differs from the single-GPU payload"
            slab = {"what": "ONE %s image cut into %d block-row slabs (astcenc_b200_compress_image_sharded): every rank uploads and searches its rows only, "
                            "grouped ncclSend/ncclRecv gather into rank 0's device buffer, one D2H; byte-identical to the single-GPU payload (checked)" % (workload_name(c).split(" (")[0], world),
                    "value": DIM * DIM / (slab_ms * 1e-3) / 1e6, "unit": "Mtexels/s", "scaling": "strong", "ms_per_image": slab_ms,
                    "search_ms_max_over_ranks": slab_search_ms, "gather_ms_max_over_ranks": slab_gather_ms,
                    "gather_bytes": payload - (payload // world), "limit": "per-rank tail waves of the search (the late waves do not fill 148 SMs) + the fixed ~30 launches per slab; the gather moves "
                    "%.1f MB and is not the limit" % ((payload - payload // world) / 1e6)}
        if e2e_s is None:
            e2e_s, images_e2e, e2e_h2d, e2e_d2h = slab_s, 1, image_bytes, payload
            e2e_mode = "astcenc_b200_compress_image_sharded (slab mode)"

    times = torch.tensor([dev_ms, e2e_s * 1e3, kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, kernel_ms = [float(x) for x in times.cpu()]

    if rank == 0:
        texels = DIM * DIM * world
        value = texels / (dev_ms * 1e-3) / 1e6
        peak, peak_kind = measured_peak_hbm()
        achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
        line = {"metric": metric, "value": value, "unit": "Mtexels/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "images_per_step": world,
                "sharding": "one image per rank per step, payload (16 B/block) gathered to rank 0 over NCCL" if world > 1 else "single GPU",
                "e2e": {"value": DIM * DIM * images_e2e / (e2e_ms * 1e-3) / 1e6, "unit": "Mtexels/s", "h2d_bytes_per_step": e2e_h2d, "d2h_bytes_per_step": e2e_d2h,
                        "ms_per_step": e2e_ms, "images_per_step": images_e2e, "path": e2e_mode, "host_memory": "pageable"},
                "gpu_launches": launches,
                "clocks": clocks,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic_from_profile() if c in (1, 4) else None,
                             "peak_source": peak_kind + " copy bandwidth (MEASURED_PEAKS.json)",
                             "kernel": "wave pipeline = astc_wave_{setup,refine,prepare,emit}_kernel, one pass over the image (%d launches)" % (launches // max(1, K)),
                             "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": algo_bytes,
                             "stage_ms": stage_ms, "stage_launches": stage_launches,
                             "dominant_kernel": "astc_wave_%s_kernel" % max(stage_ms, key=stage_ms.get),
                             "note": "achieved = (texels in + blocks out) / duration of one pipeline pass (CUDA events on the launching stream); traffic = DRAM bytes "
                                     "of the same pass from ncu, it includes the per-block records the stage kernels exchange; the search is issue/latency "
                                     "bound, not bandwidth bound - frac is reported against the HBM roofline as the tier requires"},
                "wall_ms_per_step": wall * 1e3 / K}
        if slab is not None:
            line["slab"] = slab
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(c, base)
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
