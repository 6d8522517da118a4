import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _build_once():
    import __graft_entry__ as ge
    ge.build_cpu_side()


@pytest.fixture(scope="session")
def built():
    _build_once()
    return True


@pytest.fixture(scope="session")
def port(built):
    from oracle.oracle import Oracle
    return Oracle("port")


def _golden():
    """tests/golden/make_golden.py: the stored outputs of the reference's codec and the inputs they belong to."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def pytest_report_header(config):
    from oracle.oracle import available
    if available("reference"):
        return "parity oracle: reference build (oracle/_ref/libreflz4.so)"
    return "parity oracle: restatement (oracle/lz4_oracle.c), checked first against the stored reference outputs in tests/golden"


@pytest.fixture(scope="session")
def ref(built):
    """The reference's codec where oracle/Makefile could build it into oracle/_ref (it needs the reference's source tree,
    which the repository does not contain).  Otherwise the restatement (oracle/lz4_oracle.c), and only after it has
    reproduced, byte for byte, every stored output of the reference's codec in tests/golden/golden.json and decoded it
    back (the report header says which one a run uses)."""
    from oracle.oracle import Oracle, available
    if available("reference"):
        return Oracle("reference")
    golden = _golden()
    port = Oracle("port")
    for case in golden.load("golden.json")["cases"]:
        try:
            golden.check_golden_case(port, case)
        except AssertionError as e:
            pytest.fail(f"the restatement no longer reproduces the reference's stored output ({e}): it cannot stand in "
                        "for the reference")
    return port


@pytest.fixture(scope="session")
def ctx(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from streamly_lz4_b200 import Context
    c = Context(0)
    yield c
    c.close()
