"""Shared fixtures.  `-m "not gpu"` runs on a CPU-only box; `-m gpu` needs a B200.

The checkers (oracle/) are used here only to CHECK: the product path (raytracerwin_b200) never
imports them.  The reference's compiled hot path (oracle/_ref/*.so) and its Data folder
(assets/_ref/Data) are build outputs of oracle/Makefile where the reference's sources are at hand.
Without them:
  * the scenes load generated stand-ins with the same file names (tests/standin_data.py), and the
    golden fixtures are those of the stand-ins (tests/golden/standin/);
  * the CPU tests that pin the restatement to the reference skip; the GPU tests compare the CUDA
    path with the restatement instead (tests/port_reference.py), which those CPU tests pin.
"""
import os
import sys
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DATA_DIR = os.path.join(ROOT, "assets", "_ref", "Data")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def _have_gpu():
    try:
        import raytracerwin_b200 as rt
        return rt.load_library().rt_gpu_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _have_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def rt():
    import raytracerwin_b200 as m
    m.load_library()
    return m


@pytest.fixture(scope="session")
def data_dir(tmp_path_factory):
    """Meshes for the scenes of scenes.py: the reference's Data folder where staged, else generated stand-ins."""
    if os.path.isdir(DATA_DIR):
        return DATA_DIR
    import standin_data
    return standin_data.write(str(tmp_path_factory.mktemp("standin") / "Data"))


_ORACLES = {}


def _ref_oracle(counting):
    """One RefOracle per library for the whole session."""
    from oracle import bindings
    if counting not in _ORACLES:
        _ORACLES[counting] = bindings.RefOracle(counting=counting)
    return _ORACLES[counting]


def _port_reference(request):
    """GPU tests only: the restatement in the reference's place (tests/port_reference.py)."""
    from oracle import bindings
    if request.node.get_closest_marker("gpu") is None or not bindings.port_available():
        return None
    import raytracerwin_b200
    from port_reference import PortReference
    raytracerwin_b200.load_library()
    return PortReference(raytracerwin_b200, bindings.PortOracle())


@pytest.fixture
def ref(request):
    from oracle import bindings
    if not bindings.ref_available():
        stand_in = _port_reference(request)
        if stand_in is None:
            pytest.skip("oracle/_ref/libref_oracle.so not built")
        return stand_in
    return _ref_oracle(False)


@pytest.fixture
def ref_counting(request):
    """The ray-counting twin of the reference (RayTracerScene.cpp built with -finstrument-functions): same
    results, and ref.render(...)["rays"] = the number of FindIntersectionWithScene calls it made."""
    from oracle import bindings
    if not os.path.exists(bindings.REF_COUNT_LIB):
        stand_in = _port_reference(request)       # counts the same rays (tests/test_oracle_vs_ref.py)
        if stand_in is None:
            pytest.skip("oracle/_ref/libref_oracle_count.so not built")
        return stand_in
    return _ref_oracle(True)


@pytest.fixture(scope="session")
def port():
    from oracle import bindings
    if not bindings.port_available():
        pytest.skip("oracle/librt_oracle.so not built")
    return bindings.PortOracle()


@pytest.fixture(scope="session")
def gpu(rt):
    ctx = rt.GpuContext(0)
    yield ctx
    ctx.close()


def is_reference(ref, what):
    """True where `ref` is the reference itself.  With the restatement in its place (port_reference.py), `what`
    (output of the host scene layer: loader counts, tree, unit-vector table) would be compared with itself: the
    caller leaves that comparison out, and the warning summary says so."""
    if getattr(ref, "stands_in", False):
        warnings.warn(f"{what}: not compared: no compiled reference (oracle/_ref), and the restatement in its place "
                      "shares the host scene layer under test")
        return False
    return True


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_bits(a, b):
    """Bit-identical, except that NaNs only have to coincide in position (x86 and CUDA give NaNs different
    sign/payload bits; the reference itself produces NaN radiance at a few degenerate hits)."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])
