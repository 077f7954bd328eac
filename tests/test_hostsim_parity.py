"""CPU-only parity tests: the device code compiled as a single-lane simulator (tests/hostsim) against the committed
golden GAF of the unmodified reference, and against oracle/_ref or its stored results. Exercises host logic (GFA loader,
index build, batch dispatcher, result assembly, GAF writer) and the control flow of every kernel stage."""
import pytest

import cases
import mgtest as T


@pytest.fixture(scope="module")
def lib():
    return T.load_hostsim()


def test_c1_fixture_reads(lib, workdir):
    cases.case_c1(lib, workdir)


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
    cases.case_switches(lib, workdir, device=False)


def test_upload_modes(lib, workdir):
    cases.case_upload_modes(lib, workdir)


def test_index_vs_reference_lists(lib, workdir):
    cases.case_index_big(lib, workdir, graph_len=2000000, n_probe=5000)


def test_index_on_several_devices(lib, workdir):
    import torch
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    cases.case_multi_device(lib, workdir, devices="0,1" if n >= 2 else "0,0,0")


def test_concurrent_callers(lib, workdir):
    cases.case_concurrent_calls(lib, workdir)


def test_small_max_lc_skip(lib, workdir):
    cases.case_chain_skip(lib, workdir)


def test_struct_fields_vs_reference(lib, workdir):
    cases.case_struct_random(lib, workdir, n_reads=60)


def test_graph_chaining_label_table(lib, workdir):
    cases.case_gchain_labels(lib, workdir, n_reads=150)


def test_gap_alignment_tiers(lib, workdir):
    cases.case_wfa_tiers(lib, workdir)


def test_wfa_iteration_cap_fallback(lib):
    cases.case_wfa_fallback(lib)
    cases.case_wfa_divergent(lib)
    cases.case_wfa_band_shrinks(lib)


def test_full_size_properties_small(lib, workdir):
    """the logic of the GPU suite's full-size test (tests/test_gpu_zz_full_size.py) at a size the simulator finishes"""
    cases.case_full_size(lib, workdir, n_reads=120, n_sub=40, n_ref=20)








def test_gaf_batch_writer_reuses_buffer(lib, workdir):
    """mgb_write_gaf_batch(): several threads, the caller's buffer handed back and reused, same bytes as the one-read writer"""
    import ctypes as C
    import os
    from minigraph_b200 import capi, options
    hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mt.gafw.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, 300, 2000, "ont", 41)
    names, seqs = T.read_fasta(reads)
    g = lib.mgb_gfa_read(os.path.join(T.FIX, "MT.gfa").encode())
    io, mo = options.opt_set("lr", True)
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    n = len(seqs)
    qlens = (C.c_int * n)(*[len(s) for s in seqs])
    cseqs, cnames = (C.c_char_p * n)(*seqs), (C.c_char_p * n)(*names)
    gcs = (C.POINTER(capi.mg_gchains_t) * n)()
    assert lib.mg_map_batch(gi, n, qlens, cseqs, cnames, gcs, C.byref(mo)) == 0, lib.mgb_last_error()
    one, ln1, cap1 = C.c_void_p(0), C.c_size_t(0), C.c_size_t(0)
    for i in range(n):
        lib.mgb_write_gaf(C.byref(one), C.byref(ln1), C.byref(cap1), g, gcs[i], qlens[i], cnames[i], mo.flag)
    want = C.string_at(one, ln1.value)
    buf, ln, cap = C.c_void_p(0), C.c_size_t(0), C.c_size_t(0)
    seen = set()
    for threads in (4, 7, 1, 4):
        lib.mgb_write_gaf_batch(g, n, gcs, qlens, cnames, mo.flag, threads, C.byref(buf), C.byref(ln), C.byref(cap))
        assert C.string_at(buf, ln.value) == want
        assert cap.value > ln.value
        seen.add(buf.value)
    assert len(seen) == 1  # the buffer of the first call served all of them
    fresh, lnf = C.c_void_p(0), C.c_size_t(0)
    lib.mgb_write_gaf_batch(g, n, gcs, qlens, cnames, mo.flag, 3, C.byref(fresh), C.byref(lnf), None)
    assert C.string_at(fresh, lnf.value) == want
    C.CDLL(None).free(fresh)
    lib.mgb_free_batch(n, gcs)
    assert all(not gcs[i] for i in range(n))
    lib.mg_idx_destroy(gi)


def test_exact_radix_sort_in_place_and_by_digit_walk(lib):
    cases.case_radix_exact(lib)


def test_rmq_chaining_with_interleaved_diagonals(lib, workdir):
    cases.case_tandem_diagonals(lib, workdir)
