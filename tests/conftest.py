import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def hjd():
    import hls_jpeg_decoder_b200 as pkg
    if not os.path.exists(pkg.LIB_PATH):
        pkg.build()
    return pkg


@pytest.fixture(scope="session")
def port():
    from oracle import port as p
    p.build()
    return p


@pytest.fixture(scope="session")
def refbind():
    from oracle import refbind as r
    if not r.available("std"):
        pytest.skip("oracle/_ref not built: needs a checkout of the original project, which is not part of this "
                    "repository (REF=<checkout> oracle/build_ref.sh)")
    return r
