import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _make(directory, *targets):
    subprocess.run(["make", "-C", directory, *targets], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)


@pytest.fixture(scope="session")
def emu_lib():
    """Test-only CPU emulation build of the product sources (tests/emu)."""
    from sunscreen_b200.lib import B200Lib
    _make(os.path.join(ROOT, "tests", "emu"))
    return B200Lib(os.path.join(ROOT, "tests", "emu", "_build", "libb200bfv_emu.so"), _allow_emu=True)


@pytest.fixture(scope="session")
def port():
    """The plain-C restatement of the path (oracle/bfv_oracle.c)."""
    import oracle_port
    _make(os.path.join(ROOT, "oracle"), "port")
    return oracle_port.OraclePort()


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference (oracle/_ref/libsealc_ref.so); built here when /root/reference exists,
    shipped prebuilt to the GPU box."""
    import refseal
    if os.path.exists("/root/reference/seal_fhe/SEAL/native/src/seal/seal.h"):
        _make(os.path.join(ROOT, "oracle"), "-j8", "ref")
    if not refseal.have_ref():
        pytest.skip("reference library oracle/_ref/libsealc_ref.so not available")
    return refseal.RefLib.get()


@pytest.fixture(scope="session")
def ref_or_none(request):
    """The reference library when it is available, else None: the parity checks then compare with the records of its
    outputs in tests/golden/reference_parity.json."""
    try:
        return request.getfixturevalue("ref")
    except pytest.skip.Exception:
        return None
