import gzip
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def unhex(s):
    return bytes.fromhex(s[2:] if s.startswith("0x") else s)


class Vectors:
    """c-kzg-4844 mainnet vectors shipped with the reference, converted by tests/golden/make_fixtures.py."""

    def __init__(self):
        with open(os.path.join(GOLDEN, "ckzg_vectors.json")) as fh:
            self.v = json.load(fh)
        with gzip.open(os.path.join(GOLDEN, "ckzg_blobs.bin.gz"), "rb") as fh:
            raw = fh.read()
        self.blobs, off = [], 0
        for n in self.v["blob_lengths"]:
            self.blobs.append(raw[off:off + n])
            off += n

    def __getitem__(self, k):
        return self.v[k]


@pytest.fixture(scope="session")
def vectors():
    return Vectors()


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O
    O.build()
    O.lib()
    return O
