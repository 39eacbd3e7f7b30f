import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PKG = "3d-lidar-multi-object-tracking_b200"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


@pytest.fixture(scope="session")
def pkg():
    return importlib.import_module(PKG)


@pytest.fixture(scope="session")
def synth():
    return importlib.import_module(PKG + ".synth")


# The reference's answers to the parity tests are stored in tests/golden/reference_calls.npz (oracle/recorded.py), so the tests compare
# against the reference wherever they run.  LMOT_RECORD_REFERENCE_CALLS=<path.npz> regenerates the file from oracle/_ref (built by
# build() where the reference's sources are present) while the whole suite runs on a GPU.
REFERENCE_CALLS = os.path.join(ROOT, "tests", "golden", "reference_calls.npz")
RECORD_TO = os.environ.get("LMOT_RECORD_REFERENCE_CALLS")
_streams = {}
_ports = {}
_replay = []


def _reference(request, mode):
    from oracle import recorded
    key = (f"{request.node.module.__name__}::{request.node.name}", mode)
    if mode not in _ports:                       # one restatement per mode, like the reference's process-global tracker
        _ports[mode] = recorded.private_port(mode)
    if RECORD_TO:
        _streams[key] = recorded.RecordingOracle(mode, _ports[mode])
        return _streams[key]
    if not _replay:
        _replay.append(recorded.load(REFERENCE_CALLS))
    index, calls, arrays = _replay[0]
    if key not in index:
        pytest.fail(f"no recorded reference answers for {key} in {REFERENCE_CALLS}")
    return recorded.ReplayOracle(mode, _ports[mode], calls[index[key]], arrays, index[key])


def pytest_sessionfinish(session):
    if RECORD_TO and _streams:
        from oracle import recorded
        recorded.save(RECORD_TO, _streams)


@pytest.fixture
def ref_intended(request):
    return _reference(request, "intended")


@pytest.fixture
def ref_o2(request):
    return _reference(request, "o2")


@pytest.fixture(scope="session")
def lm(pkg):
    """One liblmot context on cuda:0 for the whole GPU test session."""
    ctx = pkg.Lmot(device=0)
    yield ctx
    ctx.close()
