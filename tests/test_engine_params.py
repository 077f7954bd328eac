"""mgb_set_param() on the CPU build of the library (tests/hostsim): every key INTEGRATION.md section 4 and the switch cases use is
accepted, the launch shapes "sw<N>" / "mb<N>" keep to their bounds, and anything else is refused with -1. Every value a test sets
is put back to the library's default, since the library stays loaded for the other tests of the session."""
import pytest

import mgtest as T

DEFAULTS = {b"device": 0, b"host_threads": 0, b"slots": 3, b"slot_workers": 0, b"arena_mb": 6, b"arena_big_mb": 1024,
            b"workers_per_sm": 32, b"lab_cache": 1, b"pack2": 1, b"index_dev": 1, b"gpu_lock": 1, b"tier_learn": 1}
# launch shape of stages 0-9 (the stage table of mgb_engine.cu): warps per block ("sw<N>") and blocks per SM ("mb<N>")
WARPS = [4, 7, 4, 4, 4, 4, 2, 4, 4, 4]
BLOCKS = [8, 2, 8, 8, 5, 8, 7, 4, 4, 4]


@pytest.fixture(scope="module")
def lib():
    return T.load_hostsim()


def test_documented_keys_accepted(lib):
    for k, v in DEFAULTS.items():
        assert lib.mgb_set_param(k, v) == 0, k
    for s in (7, 8):  # tests/cases.py case_switches
        assert lib.mgb_set_param(b"sw%d" % s, WARPS[s]) == 0
        assert lib.mgb_set_param(b"mb%d" % s, BLOCKS[s]) == 0


def test_launch_shape_bounds(lib):
    for s in range(10):
        sw, mb = b"sw%d" % s, b"mb%d" % s
        for v in (-1, 0, 5, 32):
            assert lib.mgb_set_param(sw, v) == -1, (sw, v)
        for v in (-1, 0, 33):
            assert lib.mgb_set_param(mb, v) == -1, (mb, v)
        # k_chain's default of 7 warps is above what "sw1" accepts, so that one is not changed here: it could not be put back
        settable_sw = WARPS[s] <= 4
        try:
            for v in (1, 16, 32):
                assert lib.mgb_set_param(mb, v) == 0, (mb, v)
            for v in ((1, 2, 3, 4) if settable_sw else ()):
                assert lib.mgb_set_param(sw, v) == 0, (sw, v)
        finally:
            lib.mgb_set_param(mb, BLOCKS[s])
            if settable_sw:
                lib.mgb_set_param(sw, WARPS[s])


def test_unknown_keys_rejected(lib):
    for k in (b"thread_mask", b"block_warps", b"", b"arena", b"ARENA_MB", b"sw", b"mb", b"swx", b"sw10", b"mb17", b"sw19", b"mb1x"):
        assert lib.mgb_set_param(k, 1) == -1, k
