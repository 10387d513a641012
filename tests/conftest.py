import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "examples"))  # host_circuits (caller-side example package)
sys.path.insert(0, os.path.join(ROOT, "tests"))     # host_backend (test infrastructure)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # a fresh checkout has no built library (it is git-ignored): build it once, in-tree
    lib = os.path.join(ROOT, "renegade_b200", "libb200prover.so")
    if not os.path.exists(lib):
        import subprocess
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "renegade_b200", "csrc"), "-j4", "-s"])


@pytest.fixture(scope="session")
def oracle():
    """The C restatement (test infrastructure)."""
    import oracle_c
    oracle_c.build()
    return oracle_c


@pytest.fixture(scope="session")
def pyoracle():
    import bn254_py
    return bn254_py


@pytest.fixture(scope="session")
def kat():
    import json
    with open(os.path.join(ROOT, "tests", "golden", "kat.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def srs_head():
    with open(os.path.join(ROOT, "tests", "golden", "srs_head.bin"), "rb") as f:
        return f.read()


PTAU_TAU = 0xB200B200B200


@pytest.fixture(scope="session")
def ptau_2_16(oracle, pyoracle, srs_head):
    """A ptau file of 2^16 + 3 G1 powers of tau = PTAU_TAU: the 80-byte header of the reference's SRS file, then the
    records [tau^i]_1.  The tests that prove circuits of up to 2^16 gates need that many powers; the reference's own
    file is too large to store, so its first 512 powers and its G2 records are what tests/golden keeps of it."""
    tau = oracle.int_to_limbs(pyoracle.to_mont(PTAU_TAU % pyoracle.R, pyoracle.R))
    return srs_head[:80] + oracle.srs_from_tau(tau, (1 << 16) + 3).tobytes()


@pytest.fixture(scope="session")
def ptau_g2(g2_raw):
    """(h, tau * h) of ptau_2_16: the reference's h and its multiple by PTAU_TAU, 16 x uint64 each."""
    import numpy as np
    import bn254_pairing_py as pr
    h = g2_raw[0]
    tau_h = pr.g2_mul(pr.decode_g2_mont(h.tobytes(), 0), PTAU_TAU)
    return h, np.frombuffer(pr.encode_g2_mont(tau_h), dtype=np.uint64).copy()


@pytest.fixture(scope="session")
def g2_raw():
    """(h, tau * h): the two G2 records of the reference's SRS (tests/golden/srs_g2.bin), 16 x uint64 each."""
    import numpy as np
    raw = np.frombuffer(open(os.path.join(ROOT, "tests", "golden", "srs_g2.bin"), "rb").read(), dtype=np.uint64)
    return raw[:16].copy(), raw[16:32].copy()


@pytest.fixture(scope="session")
def ctx():
    """GPU context; the extension must be present — no skipping to a CPU path."""
    import renegade_b200 as rb
    c = rb.Context(0)
    yield c
    c.close()
