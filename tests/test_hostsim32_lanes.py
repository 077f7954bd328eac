"""CPU-only: the device code with a 32-lane warp simulated by fibres (minigraph_b200/csrc/mgb_simlanes.h).

The one-lane simulator (test_hostsim_parity.py) checks control flow; this build executes the ballots, prefix scans,
order-preserving compactions and lane-0 hand-overs exactly as a warp does -- with the most adversarial schedule there is
(a lane runs alone until it needs the others) -- and stops when lanes do not meet at the same helper.  Small inputs:
a simulated exchange costs 32 context switches, and every lane repeats the scalar work.  MGB_SIM_SEED=<n> in the environment
resumes the lanes in a different random order every round (other interleavings, the same results);
MGB_SIM_SEGV_TRACE=1 prints stage, item, lane and a backtrace on a crash."""
import os

import pytest

import cases
import mgtest as T

@pytest.fixture(scope="module")
def lib():
    return T.load_hostsim32()


def _same_as_reference(lib, gfa, names, seqs, preset):
    want, _ = T.map_with_ref(gfa, names, seqs, preset)
    got, _, _ = T.map_with_engine(lib, gfa, names, seqs, preset)
    n_mapped = 0
    for i, (a, b) in enumerate(zip(want, got)):
        d = T.diff_results(a, b)
        assert d is None, (names[i], d)
        n_mapped += bool(a and a["n_gc"] > 0)
    return n_mapped


def test_long_reads_on_mt_graph(lib, workdir):
    hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mt.l32.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, 4, 10000, "ont", 71)
    names, seqs = T.read_fasta(reads)
    assert _same_as_reference(lib, os.path.join(T.FIX, "MT.gfa"), names, seqs, "lr") >= 3


def test_long_reads_on_sv_graph(lib, workdir):
    pre, reads = os.path.join(workdir, "sv32"), os.path.join(workdir, "sv32.reads.fa")
    T.sim_graph(pre, 200000, 3, 7)
    T.sim_reads(pre + ".hap.fa", reads, 3, 12000, "ont", 5)
    names, seqs = T.read_fasta(reads)
    assert _same_as_reference(lib, pre + ".gfa", names, seqs, "lr") >= 2


def test_asm_preset_rmq_chaining(lib, workdir):
    reads = os.path.join(workdir, "mth32.fa")
    T.sim_reads(os.path.join(T.FIX, "MT-human.fa"), reads, 2, 8000, "hifi", 13, circular=True)
    names, seqs = T.read_fasta(reads)
    assert _same_as_reference(lib, os.path.join(T.FIX, "MT-human.fa"), names, seqs, "asm") >= 1


def test_edge_reads(lib, workdir):
    cases.case_edge(lib, workdir)


def test_multi_segment_fragments(lib, workdir):
    cases.case_multi_segment(lib, workdir, n_frag=6)


def test_short_read_preset(lib, workdir):
    cases.case_short_reads(lib, workdir, n_pairs=30)


def test_no_diag_flag(lib, workdir):
    cases.case_no_diag(lib, workdir)


def test_graph_chaining_label_table(lib, workdir):
    cases.case_gchain_labels(lib, workdir, n_reads=45, graph_len=600000)


def test_wfa_tiers_and_fallback(lib):
    cases.case_wfa_fallback(lib)
    cases.case_wfa_band_shrinks(lib)


def test_exact_radix_sort_in_place_and_by_digit_walk(lib):
    cases.case_radix_exact(lib)


def test_rmq_chaining_with_interleaved_diagonals(lib, workdir):
    cases.case_tandem_diagonals(lib, workdir)
