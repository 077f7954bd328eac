"""RMQ chaining where two diagonals interleave in target order, on the GPU (runs after everything else: added at the end of round 2 with the
two-summaries-per-block outer query of chain_rmq_fill_w; the same case runs in both CPU simulators)."""
import pytest

import cases
from minigraph_b200 import capi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    return capi.load_product()


def test_rmq_chaining_with_interleaved_diagonals(lib, workdir):
    cases.case_tandem_diagonals(lib, workdir, n_reads=200)
