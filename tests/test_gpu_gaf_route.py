"""GPU tests of mgb_map_batch_gaf() on libmgb200.so: the GAF text formatted by k_gaf_size / k_gaf_write against the host route
(mg_map_batch + mgb_write_gaf_batch) and the golden text, plus two larger batches compared as a whole."""
import pytest

import gafcases
from minigraph_b200 import capi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    return capi.load_product()


def test_golden_small(lib, workdir):
    gafcases.case_golden(lib, workdir)


def test_golden_large(lib, workdir):
    gafcases.case_golden_large(lib, workdir)


def test_flag_matrix(lib, workdir):
    gafcases.case_flags(lib, workdir)


def test_path_forms(lib, workdir):
    gafcases.case_paths(lib, workdir)


def test_rare_branches(lib, workdir):
    gafcases.case_rare(lib, workdir)


def test_write_lchain_refused(lib, workdir):
    gafcases.case_refused(lib, workdir)


def test_buffer_reuse(lib, workdir):
    gafcases.case_reuse(lib, workdir)


def test_multi_device(lib, workdir):
    import torch
    gafcases.case_multi_device(lib, workdir, devices="0,0" if torch.cuda.device_count() <= 1 else "0,1")


def test_concurrent_callers(lib, workdir):
    gafcases.case_concurrent(lib, workdir)


def test_large_arena_retry(lib, workdir):
    gafcases.case_retry(lib, workdir)


def test_2000_mt_reads(lib, workdir):
    gafcases.case_big_mt(lib, workdir)


def test_1000_reads_sv_1mb_h8(lib, workdir):
    gafcases.case_big_sv(lib, workdir)
