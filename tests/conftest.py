import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with `-m gpu` under gpurun)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle_py as op
    op.build(ref=True)
    return op


@pytest.fixture(scope="session")
def have_ref(oracle):
    if not oracle.have_ref():
        pytest.skip("oracle/_ref/libref_alglib_qp.so not built (needs /root/reference)")
    return True


@pytest.fixture(scope="session")
def emu():
    from tests import util
    return util.Emu()


@pytest.fixture(scope="session")
def oracle_qp(oracle, emu):
    """The QP solver of the live oracle's control cycle: the compiled reference ALGLIB wherever it is built (oracle/Makefile
    `make ref`).  Elsewhere the solver restatement (util.Emu.oracle_qp_fn): this project's own qp_warp.cuh built for the host, so
    there the live oracle checks the stages around the solve (dynamics, estimate, assembly, torque map) independently, while the
    solve itself is checked against the reference's stored outputs (tests/golden: qp_*.npz, cycle_*.npz).
    Tests of the reference ALGLIB itself take `have_ref`."""
    return "ref" if oracle.have_ref() else emu.oracle_qp_fn()


@pytest.fixture(scope="session")
def gpu_batch():
    """A WbcBatch on cuda:0.  Fails (not skips) when the CUDA library cannot be used: no CPU fallback."""
    from wbc_quadruped_dob_b200 import api
    b = api.WbcBatch(max_batch=70000, device=0)
    yield b
    b.close()
