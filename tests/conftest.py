import ctypes
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def cuda_device_count():
    """CUDA devices the driver reports, 0 without a driver or a device.  Asked of the driver rather than read off
    /dev/nvidia0: a container may expose its only GPU under another index, and CUDA_VISIBLE_DEVICES may hide all."""
    try:
        cuda = ctypes.CDLL("libcuda.so.1")
    except OSError:
        return 0
    n = ctypes.c_int(0)
    if cuda.cuInit(0) != 0 or cuda.cuDeviceGetCount(ctypes.byref(n)) != 0:
        return 0
    return n.value


HAS_GPU = cuda_device_count() > 0


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")
    # The shared libraries are git-ignored build products.  Build whatever is missing (g++/nvcc
    # only, no GPU needed) so a fresh checkout can run the suite.
    need = [os.path.join(ROOT, "vecchio_b200", "lib", "libvecchio_host.so"),
            os.path.join(ROOT, "vecchio_b200", "lib", "libvecchio_gpu.so"),
            os.path.join(ROOT, "vecchio_b200", "lib", "vecchio_gpu_render"),
            os.path.join(ROOT, "oracle", "liboracle.so")]
    if not all(os.path.exists(p) for p in need):
        subprocess.run(["make", "-j4", "all"], cwd=ROOT, check=True, stdout=subprocess.DEVNULL)


@pytest.fixture(scope="session")
def vb():
    import vecchio_b200
    return vecchio_b200


@pytest.fixture(scope="session")
def po():
    from oracle import pyoracle
    return pyoracle


@pytest.fixture(scope="session")
def ctx(vb):
    """One GPU context for the whole session (gpu-marked tests only)."""
    c = vb.Context(0)
    yield c
    c.close()


_SCENES = {}


def get_scene(vb, name, seed=1, param=0):
    key = (name, seed, param)
    if key not in _SCENES:
        s = vb.Scene(name, seed=seed, param=param)
        _SCENES[key] = (s, s.next_camera())
    return _SCENES[key]
