"""GPU parity tests: libmgb200.so (CUDA, sm_100a) through the C ABI against the golden GAF and the reference (oracle/_ref or its
stored results)."""
import os

import pytest

import cases
import mgtest as T
from minigraph_b200 import capi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    return capi.load_product()


def test_c1_fixture_reads(lib, workdir):
    st = cases.case_c1(lib, workdir)
    assert st.n_launches >= 3


def test_c2_mt_synthetic(lib, workdir):
    cases.case_c2(lib, workdir)


def test_c3_sv_graph(lib, workdir):
    cases.case_c3(lib, workdir)


def test_c4_asm_preset(lib, workdir):
    cases.case_c4(lib, workdir)


def test_larger_golden_sets(lib, workdir):
    cases.case_golden_large(lib, workdir)


def test_edge_reads(lib, workdir):
    cases.case_edge(lib, workdir)


def test_multi_segment_fragments(lib, workdir):
    cases.case_multi_segment(lib, workdir)


def test_short_read_preset(lib, workdir):
    cases.case_short_reads(lib, workdir)


def test_no_diag_flag(lib, workdir):
    cases.case_no_diag(lib, workdir)


def test_learned_tier_routing_keeps_results(lib, workdir):
    cases.case_tier_routing(lib, workdir)


def test_engine_switches_keep_results(lib, workdir):
    cases.case_switches(lib, workdir, device=True)


def test_upload_modes(lib, workdir):
    cases.case_upload_modes(lib, workdir)


def test_index_of_a_50mb_graph(lib, workdir):
    cases.case_index_big(lib, workdir)


def test_index_on_several_devices(lib, workdir):
    import torch
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    cases.case_multi_device(lib, workdir, devices="0,1" if n >= 2 else "0,0,0")


def test_concurrent_callers(lib, workdir):
    cases.case_concurrent_calls(lib, workdir)


def test_small_max_lc_skip(lib, workdir):
    cases.case_chain_skip(lib, workdir)


def test_struct_fields_vs_reference(lib, workdir):
    cases.case_struct_random(lib, workdir, n_reads=400)


def test_index_matches_oracle_sketch(lib):
    import subprocess
    import ctypes as C
    import os
    import test_oracle
    subprocess.check_call(["make", "-s", "-C", os.path.join(T.REPO, "oracle"), "liboracle.so"])
    orc = C.CDLL(os.path.join(T.REPO, "oracle", "liboracle.so"))
    orc.orc_sketch.restype = C.c_int64
    orc.orc_sketch.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int64]
    test_oracle.check_index(lib, orc)








def test_graph_chaining_label_table(lib, workdir):
    cases.case_gchain_labels(lib, workdir, n_reads=600, graph_len=2000000)


def test_gap_alignment_tiers(lib, workdir):
    cases.case_wfa_tiers(lib, workdir, n_struct=150)


def test_wfa_iteration_cap_fallback(lib):
    cases.case_wfa_fallback(lib, n_cases=10)
    cases.case_wfa_divergent(lib)
