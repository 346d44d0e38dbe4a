"""ctypes bindings used by the tests: the reference build (oracle/_ref, checker only) and the oracle port.

The structs mirror astcenc.h (astcenc_config :427-605, astcenc_image :613-629, astcenc_swizzle :300-313).
"""
import ctypes as C
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libastcenc_ref_avx2.so")
ORACLE_SO = os.path.join(ROOT, "oracle", "_build", "libastc_oracle.so")

PRF_LDR_SRGB, PRF_LDR, PRF_HDR_RGB_LDR_A, PRF_HDR = 0, 1, 2, 3
PRE_FASTEST, PRE_FAST, PRE_MEDIUM, PRE_THOROUGH, PRE_VERYTHOROUGH, PRE_EXHAUSTIVE = 0.0, 10.0, 60.0, 98.0, 99.0, 100.0
FLG_MAP_NORMAL, FLG_USE_DECODE_UNORM8, FLG_USE_ALPHA_WEIGHT, FLG_USE_PERCEPTUAL = 1, 2, 4, 8
FLG_DECOMPRESS_ONLY, FLG_SELF_DECOMPRESS_ONLY, FLG_MAP_RGBM = 16, 32, 64
TYPE_U8, TYPE_F16, TYPE_F32 = 0, 1, 2


class Config(C.Structure):
    _fields_ = [
        ("profile", C.c_int), ("flags", C.c_uint), ("block_x", C.c_uint), ("block_y", C.c_uint), ("block_z", C.c_uint),
        ("cw_r_weight", C.c_float), ("cw_g_weight", C.c_float), ("cw_b_weight", C.c_float), ("cw_a_weight", C.c_float),
        ("a_scale_radius", C.c_uint), ("rgbm_m_scale", C.c_float),
        ("tune_partition_count_limit", C.c_uint), ("tune_2partition_index_limit", C.c_uint),
        ("tune_3partition_index_limit", C.c_uint), ("tune_4partition_index_limit", C.c_uint),
        ("tune_block_mode_limit", C.c_uint), ("tune_refinement_limit", C.c_uint), ("tune_candidate_limit", C.c_uint),
        ("tune_2partitioning_candidate_limit", C.c_uint), ("tune_3partitioning_candidate_limit", C.c_uint),
        ("tune_4partitioning_candidate_limit", C.c_uint),
        ("tune_db_limit", C.c_float), ("tune_mse_overshoot", C.c_float),
        ("tune_2partition_early_out_limit_factor", C.c_float), ("tune_3partition_early_out_limit_factor", C.c_float),
        ("tune_2plane_early_out_limit_correlation", C.c_float), ("tune_search_mode0_enable", C.c_float),
        ("progress_callback", C.c_void_p),
    ]


class Image(C.Structure):
    _fields_ = [("dim_x", C.c_uint), ("dim_y", C.c_uint), ("dim_z", C.c_uint), ("data_type", C.c_int), ("data", C.POINTER(C.c_void_p))]


class Swizzle(C.Structure):
    _fields_ = [("r", C.c_int), ("g", C.c_int), ("b", C.c_int), ("a", C.c_int)]


class BlockInfo(C.Structure):
    _fields_ = [
        ("profile", C.c_int), ("block_x", C.c_uint), ("block_y", C.c_uint), ("block_z", C.c_uint), ("texel_count", C.c_uint),
        ("is_error_block", C.c_bool), ("is_constant_block", C.c_bool), ("is_hdr_block", C.c_bool), ("is_dual_plane_block", C.c_bool),
        ("partition_count", C.c_uint), ("partition_index", C.c_uint), ("dual_plane_component", C.c_uint),
        ("color_endpoint_modes", C.c_uint * 4), ("color_level_count", C.c_uint), ("weight_level_count", C.c_uint),
        ("weight_x", C.c_uint), ("weight_y", C.c_uint), ("weight_z", C.c_uint),
        ("color_endpoints", C.c_float * 32), ("weight_values_plane1", C.c_float * 216), ("weight_values_plane2", C.c_float * 216),
        ("partition_assignment", C.c_uint8 * 216),
    ]


def _bind(lib):
    lib.astcenc_config_init.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.c_uint, C.POINTER(Config)]
    lib.astcenc_config_init.restype = C.c_int
    lib.astcenc_context_alloc.argtypes = [C.POINTER(Config), C.c_uint, C.POINTER(C.c_void_p), C.c_void_p]
    lib.astcenc_context_alloc.restype = C.c_int
    lib.astcenc_compress_image.argtypes = [C.c_void_p, C.POINTER(Image), C.POINTER(Swizzle), C.c_void_p, C.c_size_t, C.c_uint]
    lib.astcenc_compress_image.restype = C.c_int
    lib.astcenc_decompress_image.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(Image), C.POINTER(Swizzle), C.c_uint]
    lib.astcenc_decompress_image.restype = C.c_int
    lib.astcenc_compress_reset.argtypes = [C.c_void_p]
    lib.astcenc_compress_reset.restype = C.c_int
    lib.astcenc_get_block_info.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(BlockInfo)]
    lib.astcenc_get_block_info.restype = C.c_int
    lib.astcenc_context_free.argtypes = [C.c_void_p]
    lib.astcenc_context_free.restype = None
    lib.astcenc_get_error_string.argtypes = [C.c_int]
    lib.astcenc_get_error_string.restype = C.c_char_p
    return lib


class AstcencLib:
    """Any library exporting the astcenc.h C ABI (the reference build or the B200 product)."""

    def __init__(self, path):
        self.lib = _bind(C.CDLL(path, mode=os.RTLD_LOCAL))

    def config(self, profile, bx, by, quality, flags=0, **overrides):
        cfg = Config()
        err = self.lib.astcenc_config_init(profile, bx, by, 1, quality, flags, C.byref(cfg))
        if err:
            raise RuntimeError("config_init failed: %d" % err)
        for k, v in overrides.items():
            setattr(cfg, k, v)
        return cfg

    def compress(self, img, profile, bx, by, quality, flags=0, swz=(0, 1, 2, 3), threads=1, cfg=None, **overrides):
        """img: numpy (H, W, 4) uint8 / float16 / float32. Returns bytes of blocks."""
        if cfg is None:
            cfg = self.config(profile, bx, by, quality, flags, **overrides)
        ctx = C.c_void_p()
        err = self.lib.astcenc_context_alloc(C.byref(cfg), threads, C.byref(ctx), None)
        if err:
            raise RuntimeError("context_alloc failed: %d" % err)
        try:
            return self.compress_ctx(ctx, img, bx, by, swz, threads)
        finally:
            self.lib.astcenc_context_free(ctx)

    def compress_ctx(self, ctx, img, bx, by, swz=(0, 1, 2, 3), threads=1):
        img = np.ascontiguousarray(img)
        h, w = img.shape[:2]
        dt = {np.dtype(np.uint8): TYPE_U8, np.dtype(np.float16): TYPE_F16, np.dtype(np.float32): TYPE_F32}[img.dtype]
        slices = (C.c_void_p * 1)(img.ctypes.data)
        image = Image(w, h, 1, dt, slices)
        sw = Swizzle(*swz)
        nblocks = ((w + bx - 1) // bx) * ((h + by - 1) // by)
        out = np.zeros(nblocks * 16, dtype=np.uint8)
        if threads == 1:
            err = self.lib.astcenc_compress_image(ctx, C.byref(image), C.byref(sw), out.ctypes.data, out.nbytes, 0)
            if err:
                raise RuntimeError("compress_image failed: %d" % err)
        else:
            import threading
            errs = [0] * threads

            def run(i):
                errs[i] = self.lib.astcenc_compress_image(ctx, C.byref(image), C.byref(sw), out.ctypes.data, out.nbytes, i)
            ts = [threading.Thread(target=run, args=(i,)) for i in range(threads)]
            [t.start() for t in ts]
            [t.join() for t in ts]
            if any(errs):
                raise RuntimeError("compress_image failed: %s" % errs)
            self.lib.astcenc_compress_reset(ctx)
        return out


    NP_TYPES = {TYPE_U8: np.uint8, TYPE_F16: np.float16, TYPE_F32: np.float32}

    # ---- volumes: vol is numpy (D, H, W, 4); any block size, block_z > 1 = the 3D footprints ----
    def config3(self, profile, bx, by, bz, quality, flags=0, **overrides):
        cfg = Config()
        err = self.lib.astcenc_config_init(profile, bx, by, bz, quality, flags, C.byref(cfg))
        if err:
            raise RuntimeError("config_init failed: %d" % err)
        for k, v in overrides.items():
            setattr(cfg, k, v)
        return cfg

    def compress_volume(self, vol, profile, bx, by, bz, quality, flags=0, swz=(0, 1, 2, 3), threads=1, **overrides):
        vol = np.ascontiguousarray(vol)
        d, h, w = vol.shape[:3]
        cfg = self.config3(profile, bx, by, bz, quality, flags, **overrides)
        ctx = C.c_void_p()
        err = self.lib.astcenc_context_alloc(C.byref(cfg), threads, C.byref(ctx), None)
        if err:
            raise RuntimeError("context_alloc failed: %d" % err)
        try:
            dt = _NP2TYPE[vol.dtype]
            slices = (C.c_void_p * d)(*[vol[z].ctypes.data for z in range(d)])
            image = Image(w, h, d, dt, slices)
            sw = Swizzle(*swz)
            nblocks = ((w + bx - 1) // bx) * ((h + by - 1) // by) * ((d + bz - 1) // bz)
            out = np.zeros(nblocks * 16, dtype=np.uint8)
            if threads == 1:
                err = self.lib.astcenc_compress_image(ctx, C.byref(image), C.byref(sw), out.ctypes.data, out.nbytes, 0)
                if err:
                    raise RuntimeError("compress_image failed: %d" % err)
            else:
                import threading
                errs = [0] * threads

                def run(i):
                    errs[i] = self.lib.astcenc_compress_image(ctx, C.byref(image), C.byref(sw), out.ctypes.data, out.nbytes, i)
                ts = [threading.Thread(target=run, args=(i,)) for i in range(threads)]
                [t.start() for t in ts]
                [t.join() for t in ts]
                if any(errs):
                    raise RuntimeError("compress_image failed: %s" % errs)
            return out
        finally:
            self.lib.astcenc_context_free(ctx)

    def decompress_volume(self, blocks, w, h, d, profile, bx, by, bz, out_type=TYPE_U8, flags=0, swz=(0, 1, 2, 3), quality=PRE_MEDIUM):
        cfg = self.config3(profile, bx, by, bz, quality, flags)
        ctx = C.c_void_p()
        err = self.lib.astcenc_context_alloc(C.byref(cfg), 1, C.byref(ctx), None)
        if err:
            raise RuntimeError("context_alloc failed: %d" % err)
        try:
            blocks = np.ascontiguousarray(blocks, dtype=np.uint8)
            out = np.zeros((d, h, w, 4), dtype=self.NP_TYPES[out_type])
            slices = (C.c_void_p * d)(*[out[z].ctypes.data for z in range(d)])
            image = Image(w, h, d, out_type, slices)
            sw = Swizzle(*swz)
            err = self.lib.astcenc_decompress_image(ctx, blocks.ctypes.data, blocks.nbytes, C.byref(image), C.byref(sw), 0)
            if err:
                raise RuntimeError("decompress_image failed: %d" % err)
            return out
        finally:
            self.lib.astcenc_context_free(ctx)

    def error_metrics(self, img1, img2, hdr=False, normal=False, components=4, fstop_lo=-10, fstop_hi=10):
        """astcenc_b200_compute_error_metrics (product library only)."""
        fn = self.lib.astcenc_b200_compute_error_metrics
        fn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image), C.c_int, C.c_int, C.POINTER(ErrorMetrics)]
        fn.restype = C.c_int
        cfg = self.config(PRF_LDR, 6, 6, PRE_FAST, FLG_DECOMPRESS_ONLY)
        ctx = C.c_void_p()
        err = self.lib.astcenc_context_alloc(C.byref(cfg), 1, C.byref(ctx), None)
        if err:
            raise RuntimeError("context_alloc failed: %d" % err)
        try:
            a1, s1, i1 = _image_of(img1)
            a2, s2, i2 = _image_of(img2)
            out = ErrorMetrics()
            err = fn(ctx, int(hdr), int(normal), components, C.byref(i1), C.byref(i2), fstop_lo, fstop_hi, C.byref(out))
            if err:
                raise RuntimeError("compute_error_metrics failed: %d" % err)
            return out.as_dict()
        finally:
            self.lib.astcenc_context_free(ctx)

    def block_infos(self, blocks, profile, bx, by, flags=0, quality=PRE_MEDIUM, bz=1):
        """astcenc_get_block_info of every 16-byte block; returns a list of raw struct bytes (for exact comparison)."""
        cfg = self.config(profile, bx, by, quality, flags) if bz <= 1 else self.config3(profile, bx, by, bz, quality, flags)
        ctx = C.c_void_p()
        err = self.lib.astcenc_context_alloc(C.byref(cfg), 1, C.byref(ctx), None)
        if err:
            raise RuntimeError("context_alloc failed: %d" % err)
        try:
            blocks = np.ascontiguousarray(blocks, dtype=np.uint8).reshape(-1, 16)
            out = []
            for b in blocks:
                info = BlockInfo()
                err = self.lib.astcenc_get_block_info(ctx, b.ctypes.data, C.byref(info))
                if err:
                    raise RuntimeError("get_block_info failed: %d" % err)
                out.append(bytes(info))
            return out
        finally:
            self.lib.astcenc_context_free(ctx)

    def decompress(self, blocks, w, h, profile, bx, by, out_type=TYPE_U8, flags=0, swz=(0, 1, 2, 3), quality=PRE_MEDIUM):
        """blocks: uint8 array of 16-byte blocks. Returns a numpy (h, w, 4) image of out_type; raises on API errors."""
        cfg = self.config(profile, bx, by, quality, flags)
        ctx = C.c_void_p()
        err = self.lib.astcenc_context_alloc(C.byref(cfg), 1, C.byref(ctx), None)
        if err:
            raise RuntimeError("context_alloc failed: %d" % err)
        try:
            blocks = np.ascontiguousarray(blocks, dtype=np.uint8)
            out = np.zeros((h, w, 4), dtype=self.NP_TYPES[out_type])
            slices = (C.c_void_p * 1)(out.ctypes.data)
            image = Image(w, h, 1, out_type, slices)
            sw = Swizzle(*swz)
            err = self.lib.astcenc_decompress_image(ctx, blocks.ctypes.data, blocks.nbytes, C.byref(image), C.byref(sw), 0)
            if err:
                raise RuntimeError("decompress_image failed: %d" % err)
            return out
        finally:
            self.lib.astcenc_context_free(ctx)


def have_ref():
    return os.path.exists(REF_SO)


# ---- image error metrics (astcenccli_error_metrics.cpp) -------------------------------------------------------
REF_METRICS_SO = os.path.join(ROOT, "oracle", "_ref", "libastcenc_ref_metrics.so")
_NP2TYPE = {np.dtype(np.uint8): TYPE_U8, np.dtype(np.float16): TYPE_F16, np.dtype(np.float32): TYPE_F32}
METRIC_FIELDS = ("psnr", "alpha_psnr", "rgb_psnr", "rgb_peak", "peak_psnr", "mpsnr", "log_rmse", "mean_angular_error", "worst_angular_error")


class ErrorMetrics(C.Structure):
    """struct astcenc_b200_error_metrics (include/astcenc.h) == OracleErrorMetrics (oracle/astc_error_metrics.inl)."""
    _fields_ = [(n, C.c_double) for n in METRIC_FIELDS] + [("sum_squared_error", C.c_double * 4)]

    def as_dict(self):
        d = {n: getattr(self, n) for n in METRIC_FIELDS}
        d["sum_squared_error"] = list(self.sum_squared_error)
        return d


def _image_of(arr):
    arr = np.ascontiguousarray(arr)
    h, w = arr.shape[:2]
    slices = (C.c_void_p * 1)(arr.ctypes.data)
    return arr, slices, Image(w, h, 1, _NP2TYPE[arr.dtype], slices)


def have_ref_metrics():
    return os.path.exists(REF_METRICS_SO)


def ref_error_metrics(img1, img2, hdr=False, normal=False, components=4, fstop_lo=-10, fstop_hi=10):
    """Runs the UNMODIFIED reference compute_error_metrics() and parses what it prints (4 decimals)."""
    import re, sys, tempfile
    lib = C.CDLL(REF_METRICS_SO, mode=os.RTLD_LOCAL)
    lib.ref_compute_error_metrics.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image), C.c_int, C.c_int]
    lib.ref_compute_error_metrics.restype = None
    a1, s1, i1 = _image_of(img1)
    a2, s2, i2 = _image_of(img2)
    sys.stdout.flush()
    with tempfile.TemporaryFile(mode="w+b") as tf:
        saved = os.dup(1)
        try:
            os.dup2(tf.fileno(), 1)
            lib.ref_compute_error_metrics(int(hdr), int(normal), components, C.byref(i1), C.byref(i2), fstop_lo, fstop_hi)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
        tf.seek(0)
        text = tf.read().decode()
    keys = {"PSNR (LDR-RGBA)": "psnr", "Alpha-weighted PSNR": "alpha_psnr", "PSNR (LDR-RGB)": "rgb_psnr", "PSNR (RGB norm to peak)": "peak_psnr",
            "mPSNR (RGB)": "mpsnr", "LogRMSE (RGB)": "log_rmse", "Mean Angular Error": "mean_angular_error", "Worst Angular Error": "worst_angular_error"}
    out = {}
    for line in text.splitlines():
        m = re.match(r"\s*([^:]+):\s+(-?[0-9.]+|inf|-inf|nan)", line)
        if m and m.group(1).strip() in keys:
            out[keys[m.group(1).strip()]] = float(m.group(2))
        m = re.search(r"\(peak ([0-9.eE+-]+)\)", line)
        if m:
            out["rgb_peak"] = float(m.group(1))
    if "psnr" not in out:
        out["psnr"] = out["rgb_psnr"]      # without alpha the CLI prints the one figure as "PSNR (LDR-RGB)"
    return out


def ref_lib():
    return AstcencLib(REF_SO)


# ---- the reference build's answers, recorded ---------------------------------------------------------------------
# The tests compare with the unmodified reference build through the `reference` fixture. That build is made from the
# reference's sources, which a checkout of this repository does not have, so the fixture answers from
# tests/golden/golden_reference.npz: what the build returned for every call the tests make (tests/golden/make_golden_reference.py
# records it). Each call is keyed by a hash of its method and arguments (inputs included byte for byte, the caller's thread
# count excluded: the reference's output does not depend on it). Small outputs, and the ones a test feeds on to the next
# step, are stored whole; the others as their SHA-256, which same_bytes() compares against.
REF_RECORD = os.path.join(ROOT, "tests", "golden", "golden_reference.npz")


def _feed(h, x):
    if isinstance(x, np.ndarray):
        h.update(b"a" + x.dtype.str.encode() + repr(x.shape).encode())
        h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(b"l%d" % len(x))
        for y in x:
            _feed(h, y)
    elif isinstance(x, (bool, int, float, np.integer, np.floating)):
        h.update(b"n" + repr(float(x)).encode())
    else:
        h.update(b"s" + repr(x).encode())


def call_key(method, args):
    import hashlib
    h = hashlib.sha256(method.encode())
    _feed(h, list(args))
    return h.digest()[:8]


def output_bytes(x):
    if isinstance(x, np.ndarray):
        return np.ascontiguousarray(x).tobytes()
    if isinstance(x, list):
        return b"".join(x)
    if isinstance(x, dict):
        return np.array([x.get(k, np.nan) for k in METRIC_FIELDS], dtype=np.float64).tobytes()
    return bytes(x)


def output_digest(x):
    import hashlib
    return hashlib.sha256(output_bytes(x)).digest()[:16]


class Recorded:
    """A reference output kept as its digest only."""

    def __init__(self, digest):
        self.digest = digest


def same_bytes(got, want):
    """`got` has exactly the bytes of the reference's output `want` (an array, a list of block-info structs, or a Recorded digest)."""
    if isinstance(want, Recorded):
        return output_digest(got) == want.digest
    return output_bytes(got) == output_bytes(want)


class RecordedReference:
    """Stands in for AstcencLib(REF_SO) with the calls the tests make. With `live` (an AstcencLib on the reference build)
    every call runs the build and is recorded, and save() writes the record; without it, calls are answered from the record."""

    KEEP_BYTES = 1024

    def __init__(self, path=REF_RECORD, live=None):
        self.path, self.live = path, live
        self.kept, self.digests, self.pinned, self.last = {}, {}, set(), None
        if live is None:
            z = np.load(path)
            off, blob = z["kept_off"], z["kept_blob"]
            self.kept = {bytes(k): blob[off[i]:off[i + 1]].tobytes() for i, k in enumerate(z["kept_keys"])}
            self.digests = {bytes(k): bytes(d) for k, d in zip(z["digest_keys"], z["digests"])}

    def _call(self, method, args, run):
        key = call_key(method, args)
        self.last = key
        if self.live is not None:
            out = run(self.live)
            self.kept[key] = output_bytes(out)
            return out
        if key in self.kept:
            return self.kept[key]
        if key in self.digests:
            return Recorded(self.digests[key])
        raise KeyError("%s: no recorded reference output for these arguments (tests/golden/make_golden_reference.py records them)" % method)

    def pin(self):
        """Store the last call's output whole: a test feeds it on as input."""
        self.pinned.add(self.last)

    def save(self):
        kept = {k: v for k, v in self.kept.items() if k in self.pinned or len(v) <= self.KEEP_BYTES}
        import hashlib
        digests = {k: hashlib.sha256(v).digest()[:16] for k, v in self.kept.items() if k not in kept}
        ks = sorted(kept)
        off = np.cumsum([0] + [len(kept[k]) for k in ks]).astype(np.int64)
        blob = np.frombuffer(b"".join(kept[k] for k in ks), dtype=np.uint8)
        dk = sorted(digests)
        np.savez_compressed(self.path, kept_keys=np.array([np.frombuffer(k, np.uint8) for k in ks]).reshape(-1, 8), kept_off=off, kept_blob=blob,
                            digest_keys=np.array([np.frombuffer(k, np.uint8) for k in dk]).reshape(-1, 8),
                            digests=np.array([np.frombuffer(digests[k], np.uint8) for k in dk]).reshape(-1, 16))
        return len(ks), len(dk)

    @staticmethod
    def _array(raw, dtype, shape):
        if isinstance(raw, Recorded):
            return raw
        return np.frombuffer(raw, dtype=dtype).reshape(shape).copy() if isinstance(raw, bytes) else raw

    def compress(self, img, profile, bx, by, quality, flags=0, swz=(0, 1, 2, 3), threads=1):
        raw = self._call("compress", (img, profile, bx, by, quality, flags, tuple(swz)),
                         lambda L: L.compress(img, profile, bx, by, quality, flags, swz=swz, threads=threads))
        return self._array(raw, np.uint8, (-1,))

    def compress_volume(self, vol, profile, bx, by, bz, quality, flags=0, swz=(0, 1, 2, 3), threads=1):
        raw = self._call("compress_volume", (vol, profile, bx, by, bz, quality, flags, tuple(swz)),
                         lambda L: L.compress_volume(vol, profile, bx, by, bz, quality, flags, swz=swz, threads=threads))
        return self._array(raw, np.uint8, (-1,))

    def decompress_volume(self, blocks, w, h, d, profile, bx, by, bz, out_type=TYPE_U8, flags=0, swz=(0, 1, 2, 3), quality=PRE_MEDIUM):
        raw = self._call("decompress_volume", (np.asarray(blocks, dtype=np.uint8), w, h, d, profile, bx, by, bz, out_type, flags, tuple(swz), quality),
                         lambda L: L.decompress_volume(blocks, w, h, d, profile, bx, by, bz, out_type=out_type, flags=flags, swz=swz, quality=quality))
        return self._array(raw, AstcencLib.NP_TYPES[out_type], (d, h, w, 4))

    def block_infos(self, blocks, profile, bx, by, flags=0, quality=PRE_MEDIUM, bz=1):
        raw = self._call("block_infos", (np.asarray(blocks, dtype=np.uint8), profile, bx, by, flags, quality, bz),
                         lambda L: L.block_infos(blocks, profile, bx, by, flags=flags, quality=quality, bz=bz))
        if isinstance(raw, bytes):
            n = C.sizeof(BlockInfo)
            return [raw[i:i + n] for i in range(0, len(raw), n)]
        return raw

    def config(self, profile, bx, by, quality, flags=0):
        raw = self._call("config", (profile, bx, by, quality, flags), lambda L: L.config(profile, bx, by, quality, flags))
        return Config.from_buffer_copy(raw) if isinstance(raw, bytes) else raw

    def cli_error_metrics(self, img1, img2, hdr=False, normal=False, components=4, fstop_lo=-10, fstop_hi=10):
        """What the reference command line tool prints for the pair (ref_error_metrics)."""
        raw = self._call("cli_error_metrics", (img1, img2, hdr, normal, components, fstop_lo, fstop_hi),
                         lambda L: ref_error_metrics(img1, img2, hdr=hdr, normal=normal, components=components, fstop_lo=fstop_lo, fstop_hi=fstop_hi))
        if isinstance(raw, bytes):
            v = np.frombuffer(raw, dtype=np.float64)
            return {k: float(x) for k, x in zip(METRIC_FIELDS, v) if not np.isnan(x)}
        return raw


class OracleConfig(C.Structure):
    _fields_ = [
        ("profile", C.c_int), ("flags", C.c_uint), ("block_x", C.c_uint), ("block_y", C.c_uint), ("block_z", C.c_uint),
        ("cw_r_weight", C.c_float), ("cw_g_weight", C.c_float), ("cw_b_weight", C.c_float), ("cw_a_weight", C.c_float),
        ("a_scale_radius", C.c_uint), ("rgbm_m_scale", C.c_float),
        ("tune_partition_count_limit", C.c_uint), ("tune_2partition_index_limit", C.c_uint),
        ("tune_3partition_index_limit", C.c_uint), ("tune_4partition_index_limit", C.c_uint),
        ("tune_block_mode_limit", C.c_uint), ("tune_refinement_limit", C.c_uint), ("tune_candidate_limit", C.c_uint),
        ("tune_2partitioning_candidate_limit", C.c_uint), ("tune_3partitioning_candidate_limit", C.c_uint),
        ("tune_4partitioning_candidate_limit", C.c_uint),
        ("tune_db_limit", C.c_float), ("tune_mse_overshoot", C.c_float),
        ("tune_2partition_early_out_limit_factor", C.c_float), ("tune_3partition_early_out_limit_factor", C.c_float),
        ("tune_2plane_early_out_limit_correlation", C.c_float), ("tune_search_mode0_enable", C.c_float),
    ]


class Oracle:
    def __init__(self, path=ORACLE_SO):
        lib = C.CDLL(path)
        lib.oracle_context_create.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_float, C.c_uint, C.POINTER(C.c_float)]
        lib.oracle_context_create.restype = C.c_void_p
        lib.oracle_context_destroy.argtypes = [C.c_void_p]
        lib.oracle_compress_image.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_int), C.c_void_p]
        lib.oracle_compress_image.restype = C.c_int
        lib.oracle_get_config.argtypes = [C.c_void_p, C.POINTER(OracleConfig)]
        lib.oracle_decompress_image.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_int)]
        lib.oracle_decompress_image.restype = C.c_int
        self.lib = lib

    def error_metrics(self, img1, img2, hdr=False, normal=False, components=4, fstop_lo=-10, fstop_hi=10):
        a1 = np.ascontiguousarray(img1)
        a2 = np.ascontiguousarray(img2)
        out = ErrorMetrics()
        self.lib.oracle_error_metrics.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_uint, C.c_uint,
                                                  C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.c_int, C.c_int, C.POINTER(ErrorMetrics)]
        self.lib.oracle_error_metrics.restype = C.c_int
        err = self.lib.oracle_error_metrics(int(hdr), int(normal), components, a1.ctypes.data, _NP2TYPE[a1.dtype], a1.shape[1], a1.shape[0],
                                            a2.ctypes.data, _NP2TYPE[a2.dtype], a2.shape[1], a2.shape[0], fstop_lo, fstop_hi, C.byref(out))
        if err:
            raise RuntimeError("oracle_error_metrics failed: %d" % err)
        return out.as_dict()

    def decompress(self, blocks, w, h, profile, bx, by, out_type=TYPE_U8, flags=0, swz=None, quality=PRE_MEDIUM):
        ctx = self.lib.oracle_context_create(profile, bx, by, quality, flags, None)
        if not ctx:
            raise RuntimeError("oracle context failed")
        try:
            blocks = np.ascontiguousarray(blocks, dtype=np.uint8)
            out = np.zeros((h, w, 4), dtype=AstcencLib.NP_TYPES[out_type])
            sw = (C.c_int * 4)(*swz) if swz is not None else None
            self.lib.oracle_decompress_image(ctx, blocks.ctypes.data, out.ctypes.data, out_type, w, h, sw)
            return out
        finally:
            self.lib.oracle_context_destroy(ctx)

    def compress(self, img, profile, bx, by, quality, flags=0, swz=None, partition_count_limit=0, plane2_correlation=-1.0, a_scale_radius=0):
        img = np.ascontiguousarray(img)
        h, w = img.shape[:2]
        dt = {np.dtype(np.uint8): TYPE_U8, np.dtype(np.float16): TYPE_F16, np.dtype(np.float32): TYPE_F32}[img.dtype]
        ov = (C.c_float * 3)(float(partition_count_limit), float(plane2_correlation), float(a_scale_radius))
        ctx = self.lib.oracle_context_create(profile, bx, by, quality, flags, ov)
        if not ctx:
            raise RuntimeError("oracle context failed")
        try:
            nblocks = ((w + bx - 1) // bx) * ((h + by - 1) // by)
            out = np.zeros(nblocks * 16, dtype=np.uint8)
            sw = (C.c_int * 4)(*swz) if swz is not None else None
            self.lib.oracle_compress_image(ctx, img.ctypes.data, dt, w, h, sw, out.ctypes.data)
            return out
        finally:
            self.lib.oracle_context_destroy(ctx)

    def compress_volume(self, vol, profile, bx, by, bz, quality, flags=0, swz=None):
        vol = np.ascontiguousarray(vol)
        d, h, w = vol.shape[:3]
        self.lib.oracle_context_create_3d.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.c_uint]
        self.lib.oracle_context_create_3d.restype = C.c_void_p
        self.lib.oracle_compress_volume.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_int), C.c_void_p]
        ctx = self.lib.oracle_context_create_3d(profile, bx, by, bz, quality, flags)
        if not ctx:
            raise RuntimeError("oracle context failed")
        try:
            nblocks = ((w + bx - 1) // bx) * ((h + by - 1) // by) * ((d + bz - 1) // bz)
            out = np.zeros(nblocks * 16, dtype=np.uint8)
            sw = (C.c_int * 4)(*swz) if swz is not None else None
            self.lib.oracle_compress_volume(ctx, vol.ctypes.data, _NP2TYPE[vol.dtype], w, h, d, sw, out.ctypes.data)
            return out
        finally:
            self.lib.oracle_context_destroy(ctx)

    def decompress_volume(self, blocks, w, h, d, profile, bx, by, bz, out_type=TYPE_U8, flags=0, swz=None, quality=PRE_MEDIUM):
        self.lib.oracle_context_create_3d.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.c_uint]
        self.lib.oracle_context_create_3d.restype = C.c_void_p
        self.lib.oracle_decompress_volume.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_int)]
        ctx = self.lib.oracle_context_create_3d(profile, bx, by, bz, quality, flags)
        if not ctx:
            raise RuntimeError("oracle context failed")
        try:
            blocks = np.ascontiguousarray(blocks, dtype=np.uint8)
            out = np.zeros((d, h, w, 4), dtype=AstcencLib.NP_TYPES[out_type])
            sw = (C.c_int * 4)(*swz) if swz is not None else None
            self.lib.oracle_decompress_volume(ctx, blocks.ctypes.data, out.ctypes.data, out_type, w, h, d, sw)
            return out
        finally:
            self.lib.oracle_context_destroy(ctx)

    def config(self, profile, bx, by, quality, flags=0):
        ctx = self.lib.oracle_context_create(profile, bx, by, quality, flags, None)
        cfg = OracleConfig()
        self.lib.oracle_get_config(ctx, C.byref(cfg))
        self.lib.oracle_context_destroy(ctx)
        return cfg


def block_diff(a, b):
    """Indices of 16-byte blocks that differ."""
    a = np.asarray(a).reshape(-1, 16)
    b = np.asarray(b).reshape(-1, 16)
    return np.nonzero((a != b).any(axis=1))[0]
