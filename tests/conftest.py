import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    if r.returncode != 0:
        raise RuntimeError("%s failed:\n%s\n%s" % (cmd, r.stdout[-3000:], r.stderr[-3000:]))


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle (oracle/astc_*.cpp compiled on demand)."""
    import astc_ref
    if not os.path.exists(astc_ref.ORACLE_SO):
        _run(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"])
    return astc_ref.Oracle()


@pytest.fixture(scope="session")
def reference():
    """The unmodified reference build's answers to the tests' calls, recorded in tests/golden/golden_reference.npz."""
    import astc_ref
    return astc_ref.RecordedReference()


@pytest.fixture(scope="session")
def reference_build():
    """The unmodified reference build itself (oracle/_ref): only where oracle/Makefile could build it from the reference's sources."""
    import astc_ref
    if not astc_ref.have_ref():
        pytest.skip("reference build not available")
    return astc_ref.ref_lib()


@pytest.fixture(scope="session")
def pkg():
    import __graft_entry__ as g
    p = g.load_package()
    if not os.path.exists(p.LIB_PATH):
        p.build()
    return p


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    return np.load(os.path.join(HERE, "golden", "golden_blocks.npz"))


def _hostsim_sources():
    srcs = [os.path.join(HERE, "hostsim", "hostsim.cpp"), os.path.join(ROOT, "astc-encoder_b200", "csrc", "astc_host_tables.cpp"),
            os.path.join(ROOT, "astc-encoder_b200", "csrc", "astc_host_config.cpp")]
    csrc = os.path.join(ROOT, "astc-encoder_b200", "csrc")
    newest = max([os.path.getmtime(os.path.join(csrc, f)) for f in os.listdir(csrc)] +
                 [os.path.getmtime(os.path.join(HERE, "hostsim", f)) for f in os.listdir(os.path.join(HERE, "hostsim"))])
    return srcs, newest


@pytest.fixture(scope="session")
def hostsim32():
    """Host build of the device source with the 32 lanes of a warp emulated by 32 threads (tests/hostsim/simt_emul.h)."""
    import ctypes as C
    so = os.path.join(HERE, "_build", "libhostsim32.so")
    srcs, newest = _hostsim_sources()
    if not os.path.exists(so) or os.path.getmtime(so) < newest:
        os.makedirs(os.path.dirname(so), exist_ok=True)
        _run(["g++", "-std=c++14", "-O2", "-fPIC", "-pthread", "-ffp-contract=off", "-fno-fast-math", "-DASTC_HOSTSIM_LANES32=1", "-shared", "-x", "c++"] + srcs + ["-o", so])
    lib = C.CDLL(so)
    lib.hostsim_compress_image.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_float, C.c_uint, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_int), C.c_void_p]
    lib.hostsim_decompress_image.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_int)]
    lib.hostsim_set_a_scale_radius.argtypes = [C.c_uint]
    assert lib.hostsim_lanes() == 32
    return lib


@pytest.fixture(scope="session")
def lanes32_tsan():
    """The same simulation as a stand-alone ThreadSanitizer binary (tests/hostsim/lanes32_main.cpp); None if TSan is unavailable."""
    exe = os.path.join(HERE, "_build", "lanes32_tsan")
    srcs, newest = _hostsim_sources()
    if not os.path.exists(exe) or os.path.getmtime(exe) < newest:
        os.makedirs(os.path.dirname(exe), exist_ok=True)
        r = subprocess.run(["g++", "-std=c++14", "-O1", "-g", "-fsanitize=thread", "-fno-omit-frame-pointer", "-pthread", "-ffp-contract=off", "-fno-fast-math",
                            "-DASTC_HOSTSIM_LANES32=1", "-x", "c++", os.path.join(HERE, "hostsim", "lanes32_main.cpp")] + srcs + ["-o", exe],
                           capture_output=True, text=True)
        if r.returncode != 0:
            return None
    return exe


@pytest.fixture(scope="session")
def hostsim():
    """Host build of the device source with one simulated lane (tests/hostsim)."""
    import ctypes as C
    so = os.path.join(HERE, "_build", "libhostsim.so")
    srcs = [os.path.join(HERE, "hostsim", "hostsim.cpp"), os.path.join(ROOT, "astc-encoder_b200", "csrc", "astc_host_tables.cpp"),
            os.path.join(ROOT, "astc-encoder_b200", "csrc", "astc_host_config.cpp")]
    csrc = os.path.join(ROOT, "astc-encoder_b200", "csrc")
    newest = max([os.path.getmtime(os.path.join(csrc, f)) for f in os.listdir(csrc)] + [os.path.getmtime(srcs[0])])
    if not os.path.exists(so) or os.path.getmtime(so) < newest:
        os.makedirs(os.path.dirname(so), exist_ok=True)
        _run(["g++", "-std=c++14", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-x", "c++"] + srcs + ["-o", so])
    lib = C.CDLL(so)
    lib.hostsim_compress_image.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_float, C.c_uint, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_int), C.c_void_p]
    lib.hostsim_arena_bytes.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_float, C.c_uint]
    lib.hostsim_arena_bytes.restype = C.c_uint
    lib.hostsim_set_a_scale_radius.argtypes = [C.c_uint]
    lib.hostsim_decompress_image.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_int)]
    return lib
