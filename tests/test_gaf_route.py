"""CPU tests of mgb_map_batch_gaf(), the GAF text formatted on the device: the single-lane simulator (tests/hostsim) runs every
case, the 32-lane one (the warp's prefix sums and lane-parallel copies) the small ones.  The text must be what mg_map_batch() +
mgb_write_gaf_batch() print, byte for byte, and the golden text where there is one."""
import pytest

import gafcases
import mgtest as T


@pytest.fixture(scope="module", params=["lanes1", "lanes32"])
def lib(request):
    return T.load_hostsim() if request.param == "lanes1" else T.load_hostsim32()


@pytest.fixture(scope="module")
def lib1():
    return T.load_hostsim()


def test_golden_small(lib, workdir):
    gafcases.case_golden(lib, workdir)


def test_golden_large(lib1, workdir):
    gafcases.case_golden_large(lib1, workdir)


def test_flag_matrix(lib1, workdir):
    gafcases.case_flags(lib1, workdir)


def test_flag_matrix_lanes32(workdir):
    gafcases.case_flags(T.load_hostsim32(), workdir, flags=[gafcases.capi.MG_M_PRINT_2ND | gafcases.capi.MG_M_SHOW_UNMAP], presets=("lr",))


def test_path_forms(lib, workdir):
    gafcases.case_paths(lib, workdir)


def test_rare_branches(lib, workdir):
    gafcases.case_rare(lib, workdir)


def test_write_lchain_refused(lib, workdir):
    gafcases.case_refused(lib, workdir)


def test_buffer_reuse(lib, workdir):
    gafcases.case_reuse(lib, workdir)


def test_multi_device(lib1, workdir):
    gafcases.case_multi_device(lib1, workdir)


def test_concurrent_callers(lib1, workdir):
    gafcases.case_concurrent(lib1, workdir)


def test_large_arena_retry(lib1, workdir):
    gafcases.case_retry(lib1, workdir)
