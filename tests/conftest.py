import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def reference_strategy_dir():
    """The original project's shipped strategy XML files, stored verbatim as test data."""
    return os.path.join(ROOT, "tests", "golden", "reference_strategy")


# The reference's 4-GPU sample strategy (same topology as tests/golden/reference_strategy/4.xml), including
# its malformed attribute list `id='1'ip='...'` (no separating space) that only tinyxml2 accepts.
STRATEGY_4 = """<trees>
    <root id='0' ip='10.0.0.1'>
        <gpu id='1'ip='10.0.0.1'/>
        <gpu id='2' ip='10.0.0.1'>
            <gpu id='3' ip='10.0.0.1'/>
        </gpu>
    </root>
    <root id='2' ip='10.0.0.1'>
        <gpu id='3' ip='10.0.0.1'/>
        <gpu id='1' ip='10.0.0.1'>
            <gpu id='0' ip='10.0.0.1'/>
        </gpu>
    </root>
    <root id='3' ip='10.0.0.1'>
        <gpu id='2' ip='10.0.0.1'/>
        <gpu id='0' ip='10.0.0.1'>
            <gpu id='1' ip='10.0.0.1'/>
        </gpu>
    </root>
    <root id='1' ip='10.0.0.1'>
        <gpu id='0' ip='10.0.0.1'/>
        <gpu id='3' ip='10.0.0.1'>
            <gpu id='2' ip='10.0.0.1'/>
        </gpu>
    </root>
</trees>"""

# tree 0<-1<-{2,3} used by the reference's golden logs (log/primitive, log/training)
STRATEGY_TEST = """<?xml version="1.0" encoding="utf-8"?>
<trees>
    <root id="0" ip="10.0.0.2">
        <gpu id="1" ip="10.0.0.2">
            <gpu id="2" ip="10.0.0.2"/>
            <gpu id="3" ip="10.0.0.2"/>
        </gpu>
    </root>
    <root id="3" ip="10.0.0.2">
        <gpu id="2" ip="10.0.0.2">
            <gpu id="1" ip="10.0.0.2"/>
            <gpu id="0" ip="10.0.0.2"/>
        </gpu>
    </root>
</trees>"""


@pytest.fixture
def strategy4_xml():
    return STRATEGY_4


@pytest.fixture
def strategy_test_xml():
    return STRATEGY_TEST


def free_port() -> int:
    """A TCP port that is free right now (rendezvous ports of the multi-process CPU tests)."""
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]
