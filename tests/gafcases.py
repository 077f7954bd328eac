"""Cases of the text route, mgb_map_batch_gaf(), shared by the CPU (hostsim) and GPU (libmgb200) test modules.

Every case compares the text the call returns with what mg_map_batch() + mgb_write_gaf_batch() give on the same library
(mgtest.gaf_with_engine), and with the golden files where there are some."""
import ctypes as C
import hashlib
import os
import random
import threading

import cases
import mgtest as T
from minigraph_b200 import capi, options

MT = os.path.join(T.FIX, "MT.gfa")
MTH = os.path.join(T.FIX, "MT-human.fa")


def _arrays(names, seqs):
    n = len(seqs)
    qlens = (C.c_int * n)(*[len(s) for s in seqs])
    cseqs = (C.c_char_p * n)(*seqs)
    cnames = None if names is None else (C.c_char_p * n)(*names)
    return n, qlens, cseqs, cnames


def call_gaf(lib, gi, mo, names, seqs, buf=None, cap=None):
    """one mgb_map_batch_gaf() call: (rc, text, buf, cap, stats); buf/cap: a buffer to reuse (ownership stays with the caller)"""
    n, qlens, cseqs, cnames = _arrays(names, seqs)
    out, ln, cp = C.c_void_p(buf), C.c_size_t(0), C.c_size_t(cap or 0)
    rc = lib.mgb_map_batch_gaf(gi, n, qlens, cseqs, cnames, C.byref(mo), C.byref(out), C.byref(ln), C.byref(cp))
    text = C.string_at(out, ln.value) if out.value and ln.value else b""
    st = capi.mgb_stats_t()
    lib.mgb_get_stats(gi, C.byref(st))
    return rc, text, out.value, cp.value, ln.value, st


def free(p):
    if p:
        C.CDLL(None).free(C.c_void_p(p))


class Index:
    """mgb_gfa_read + mg_index with a preset's options, destroyed on exit"""
    def __init__(self, lib, gfa, preset="lr", cigar=True, flag_extra=0):
        self.lib = lib
        self.g = lib.mgb_gfa_read(gfa.encode())
        assert self.g, "gfa read failed"
        self.io, self.mo = options.opt_set(preset, cigar)
        self.mo.flag |= flag_extra
        self.gi = lib.mg_index(self.g, C.byref(self.io), 1, C.byref(self.mo))
        assert self.gi, lib.mgb_last_error()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.lib.mg_idx_destroy(self.gi)
        self.lib.mgb_gfa_destroy(self.g)


def gaf_route(lib, gfa, names, seqs, preset="lr", flag_extra=0, cigar=True, stats=False):
    """the text of mgb_map_batch_gaf() (names may be None: a NULL array)"""
    with Index(lib, gfa, preset, cigar, flag_extra) as ix:
        rc, text, buf, _, _, st = call_gaf(lib, ix.gi, ix.mo, names, seqs)
        free(buf)
    assert rc == 0, (rc, lib.mgb_last_error())
    return (text, st) if stats else text


def check(lib, gfa, names, seqs, preset="lr", flag_extra=0, cigar=True, want=None):
    """the route's text equals the host route's (and `want`); returns it"""
    got, st = gaf_route(lib, gfa, names, seqs, preset, flag_extra, cigar, stats=True)
    host, _ = T.gaf_with_engine(lib, gfa, [None] * len(seqs) if names is None else names, seqs, preset, cigar, flag_extra)
    assert got == host, "flag %#x cigar %d: %s" % (flag_extra, cigar, cases.first_diff(got, host))
    if want is not None:
        assert got == want, cases.first_diff(got, want)
    return got, st


def check_fasta(lib, gfa, fasta, preset="lr", want=None, flag_extra=0):
    names, seqs = T.read_fasta(fasta)
    return check(lib, gfa, names, seqs, preset, flag_extra, want=want)


# ---- 1. golden text through the new call ----
def case_golden(lib, workdir, which=("c1", "c2", "c3", "c4")):
    if "c1" in which:
        got, st = check_fasta(lib, MT, os.path.join(T.FIX, "MT-orangA.fa"), want=cases.golden("c1_MT_orangA.lr.gaf"))
        assert hashlib.md5(got).hexdigest() == "22bf23ebe2039e8353f56f4a324a2eaa"
        assert st.t_gaf_ms > 0 and st.out_bytes > 0
        check_fasta(lib, MT, os.path.join(T.FIX, "MT-chimp.fa"), want=cases.golden("c1_MT_chimp.lr.gaf"))
    if "c2" in which:
        hap, reads = os.path.join(workdir, "g_mt.hap.fa"), os.path.join(workdir, "g_mt.reads.fa")
        T.sim_mt_haps(hap)
        T.sim_reads(hap, reads, 24, 10000, "ont", 11)
        check_fasta(lib, MT, reads, want=cases.golden("c2_MT_24x10k_ont_s11.lr.gaf"))
    if "c3" in which:
        pre, reads = os.path.join(workdir, "g_sv"), os.path.join(workdir, "g_sv.reads.fa")
        T.sim_graph(pre, 300000, 3, 7)
        T.sim_reads(pre + ".hap.fa", reads, 24, 15000, "ont", 5)
        check_fasta(lib, pre + ".gfa", reads, want=cases.golden("c3_sv300k_h3_s7_24x15k_ont_s5.lr.gaf"))
    if "c4" in which:
        reads = os.path.join(workdir, "g_mth.reads.fa")
        T.sim_reads(MTH, reads, 12, 20000, "hifi", 13, circular=True)
        check_fasta(lib, MTH, reads, "asm", want=cases.golden("c4_MThuman_12x20k_hifi_s13.asm.gaf"))


def case_golden_large(lib, workdir, which=("L2", "L3", "L4")):
    if "L2" in which:
        hap, reads = os.path.join(workdir, "g_mt.hap.fa"), os.path.join(workdir, "g_mtL.reads.fa")
        T.sim_mt_haps(hap)
        T.sim_reads(hap, reads, 240, 10000, "ont", 111)
        check_fasta(lib, MT, reads, want=cases.golden_gz("L2_MT_240x10k_ont_s111.lr.gaf.gz"))
    if "L3" in which:
        pre, reads = os.path.join(workdir, "g_svL"), os.path.join(workdir, "g_svL.reads.fa")
        T.sim_graph(pre, 1000000, 8, 7)
        T.sim_reads(pre + ".hap.fa", reads, 240, 15000, "ont", 105)
        got, _ = check_fasta(lib, pre + ".gfa", reads)
        want = cases.golden("L3_sv1m_h8_s7_240x15k_ont_s105.lr.gaf.b2").split()
        lines = got.split(b"\n")
        assert lines[-1] == b"" and len(lines) - 1 == len(want)
        for i, (ln, w) in enumerate(zip(lines, want)):
            assert hashlib.blake2b(ln, digest_size=8).hexdigest().encode() == w, "line %d: %r" % (i, ln[:200])
    if "L4" in which:
        reads = os.path.join(workdir, "g_mthL.reads.fa")
        T.sim_reads(MTH, reads, 200, 20000, "hifi", 113, circular=True)
        check_fasta(lib, MTH, reads, "asm", want=cases.golden_gz("L4_MThuman_200x20k_hifi_s113.asm.gaf.gz"))


# ---- 2. flag matrix ----
FLAGS = [0, capi.MG_M_PRINT_2ND, capi.MG_M_VERTEX_COOR, capi.MG_M_NO_COMP_PATH, capi.MG_M_SHOW_UNMAP,
         capi.MG_M_PRINT_2ND | capi.MG_M_SHOW_UNMAP | capi.MG_M_NO_COMP_PATH]


def sv_graph(workdir, n_reads=24, length=9000):
    """a small SV graph with 4 haplotypes (rank > 0 segments) and reads from its haplotypes, plus two reads from nowhere"""
    pre, reads = os.path.join(workdir, "gf_sv"), os.path.join(workdir, "gf_sv.reads.fa")
    if not os.path.exists(reads):
        T.sim_graph(pre, 200000, 4, 13)
        T.sim_reads(pre + ".hap.fa", reads, n_reads, length, "ont", 17)
    names, seqs = T.read_fasta(reads)
    rnd = random.Random(3)
    names += [b"nowhere1", b"nowhere2"]
    seqs += [bytes(rnd.choice(b"ACGT") for _ in range(3000)), b"ACGTAC"]
    return pre + ".gfa", names, seqs


def case_flags(lib, workdir, flags=FLAGS, presets=("lr", "asm")):
    gfa, names, seqs = sv_graph(workdir)
    _, hs = T.read_fasta(MTH)
    mt_names, mt_seqs = [b"h%d" % i for i in range(6)], [hs[0][i * 2500:i * 2500 + 6000] for i in range(6)]
    seen = set()
    for flag in flags:
        for cigar in (True, False):
            if "lr" in presets:
                got, _ = check(lib, gfa, names, seqs, "lr", flag, cigar)
                seen.update(f for f in (b"cg:Z:", b"ds:Z:", b"\t*\t*\t") if f in got)
            if "asm" in presets:
                check(lib, MTH, mt_names, mt_seqs, "asm", flag, cigar)
    if flags is FLAGS:
        assert seen == {b"cg:Z:", b"ds:Z:", b"\t*\t*\t"}, seen


# ---- 3. path forms ----
def case_paths(lib, workdir):
    """segments without stable IDs (MT.gfa stripped of SN/SO/SR: every path is a '>name' list), and the SV graph, whose rank > 0
    segments break compaction into '>sname:st-en' runs"""
    plain = os.path.join(workdir, "gp_MT_plain.gfa")
    with open(MT) as f, open(plain, "w") as o:
        for ln in f:
            t = ln.rstrip("\n").split("\t")
            if t[0] == "S":
                t = t[:3] + [x for x in t[3:] if x[:3] not in ("SN:", "SO:", "SR:")]
            o.write("\t".join(t) + "\n")
    names, seqs = T.read_fasta(os.path.join(T.FIX, "MT-orangA.fa"))
    got, _ = check(lib, plain, names, seqs)
    assert b"\t>MT" in got or b"\t<MT" in got, got[:300]
    gfa, names, seqs = sv_graph(workdir)
    got, _ = check(lib, gfa, names, seqs)
    assert b":" in b"".join(ln.split(b"\t")[5] for ln in got.split(b"\n") if ln), "no stable-coordinate run in the paths"


# ---- 4. reads for the rare branches ----
def _rc(s):
    return s[::-1].translate(bytes.maketrans(b"ACGTN", b"TGCAN"))


def case_rare(lib, workdir):
    _, hs = T.read_fasta(MTH)
    h = hs[0]
    chim = _rc(h[2000:10000]) + h[11000:15000]  # a '-' record, then a '+' one: the sticky rev_sign reverses the second's cg and ds
    exact = h[5000:9000]                          # no error: dv:f:0
    names, seqs = [b"chimera", b"exact", b"fwd"], [chim, exact, h[300:5300]]
    got, _ = check(lib, MTH, names, seqs, "lr")
    lines = [ln.split(b"\t") for ln in got.split(b"\n") if ln.startswith(b"chimera")]
    assert [ln[4] for ln in lines][:2] == [b"-", b"+"], [ln[4] for ln in lines]
    assert b"\tdv:f:0\t" in got
    check(lib, MTH, names, seqs, "lr", capi.MG_M_PRINT_2ND)
    # empty, tiny, all-N and random reads, shown unmapped
    edge_names = [b"empty", b"tiny", b"allN", b"random", b"short_ok", b"with_N"]
    edge = [b"", b"ACGT", b"N" * 500, (b"ACGTTGCA" * 200)[:1500], h[1000:1300], h[2900:3300]]
    got, _ = check(lib, MT, edge_names, edge, "lr", capi.MG_M_SHOW_UNMAP)
    assert got.startswith(b"empty\t0\t0\t0\t*\t*\t0\t0\t0\t0\t0\t0\n"), got[:100]
    # names == NULL, and one NULL name
    got, _ = check(lib, MT, None, seqs[1:] + edge, "lr", capi.MG_M_SHOW_UNMAP)
    assert got.startswith(b"*\t")
    got, _ = check(lib, MT, [b"a", None, b"c"], [h[100:4000], h[4000:8000], b""], "lr", capi.MG_M_SHOW_UNMAP)
    assert b"\n*\t" in got


# ---- 5. -S / --write-mz refused ----
def case_refused(lib, workdir):
    _, hs = T.read_fasta(MTH)
    for bad in (capi.MG_M_WRITE_LCHAIN, capi.MG_M_WRITE_LCHAIN | capi.MG_M_WRITE_MZ):
        with Index(lib, MT, "lr", True, bad) as ix:
            rc, text, buf, _, ln, _ = call_gaf(lib, ix.gi, ix.mo, [b"r"], [hs[0][:5000]])
            free(buf)
            assert rc < 0 and ln == 0 and text == b"", (rc, ln)
            assert b"write-mz" in lib.mgb_last_error()


# ---- 6. buffer reuse ----
def case_reuse(lib, workdir):
    _, hs = T.read_fasta(MTH)
    names, seqs = [b"r%d" % i for i in range(8)], [hs[0][i * 1500:i * 1500 + 5000] for i in range(8)]
    with Index(lib, MT) as ix:
        rc, t1, buf, cap, _, _ = call_gaf(lib, ix.gi, ix.mo, names, seqs)
        assert rc == 0 and t1 and cap > len(t1)
        rc, t2, buf2, cap2, _, _ = call_gaf(lib, ix.gi, ix.mo, names[:4], seqs[:4], buf, cap)
        assert rc == 0 and buf2 == buf and cap2 == cap, "a text that fits must reuse the caller's buffer"
        assert t1.startswith(t2) and t2
        rc, t3, buf3, cap3, _, _ = call_gaf(lib, ix.gi, ix.mo, [], [], buf2, cap2)
        assert rc == 0 and t3 == b"" and buf3 == buf2
        free(buf3)


# ---- 7. several devices ----
def case_multi_device(lib, workdir, devices="0,0,0", n_reads=100):
    pre, reads = os.path.join(workdir, "gm_sv"), os.path.join(workdir, "gm_sv.reads.fa")
    T.sim_graph(pre, 300000, 3, 31)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 7000, "ont", 71)
    names, seqs = T.read_fasta(reads)
    one = gaf_route(lib, pre + ".gfa", names, seqs)
    os.environ["MGB_DEVICES"] = devices
    try:
        many = gaf_route(lib, pre + ".gfa", names, seqs)
    finally:
        del os.environ["MGB_DEVICES"]
    assert one.count(b"\n") > n_reads // 2
    assert many == one, cases.first_diff(many, one)


# ---- 8. concurrent callers ----
def case_concurrent(lib, workdir, n_threads=3, n_reads=60):
    pre, reads = os.path.join(workdir, "gc_sv"), os.path.join(workdir, "gc_sv.reads.fa")
    T.sim_graph(pre, 300000, 4, 23)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 8000, "ont", 61)
    names, seqs = T.read_fasta(reads)
    with Index(lib, pre + ".gfa") as ix:
        rc, whole, buf, _, _, _ = call_gaf(lib, ix.gi, ix.mo, names, seqs)
        free(buf)
        assert rc == 0
        out = {}

        def run(t):
            rc, text, buf, _, _, _ = call_gaf(lib, ix.gi, ix.mo, names, seqs)
            free(buf)
            out[t] = (rc, text)
        th = [threading.Thread(target=run, args=(t,)) for t in range(n_threads)]
        for x in th:
            x.start()
        for x in th:
            x.join()
    assert len(out) == n_threads
    for t, (rc, text) in out.items():
        assert rc == 0 and text == whole, "caller %d: %s" % (t, cases.first_diff(text, whole))


# ---- 9. the large-arena retry pass ----
def case_retry(lib, workdir, arena_mb=0):
    pre, reads = os.path.join(workdir, "gr_sv"), os.path.join(workdir, "gr_sv.reads.fa")
    T.sim_graph(pre, 300000, 3, 37)
    T.sim_reads(pre + ".hap.fa", reads, 12, 15000, "ont", 41)
    names, seqs = T.read_fasta(reads)
    want = gaf_route(lib, pre + ".gfa", names, seqs)
    assert lib.mgb_set_param(b"arena_mb", arena_mb) == 0
    try:
        got, st = gaf_route(lib, pre + ".gfa", names, seqs, stats=True)
    finally:
        lib.mgb_set_param(b"arena_mb", 6)
    assert st.n_retry > 0, "no read took the large-arena pass"
    assert got == want, cases.first_diff(got, want)


# ---- larger batches (GPU) ----
def case_big_mt(lib, workdir, n_reads=2000):
    hap, reads = os.path.join(workdir, "gb_mt.hap.fa"), os.path.join(workdir, "gb_mt.reads.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, n_reads, 10000, "ont", 211)
    check_fasta(lib, MT, reads)


def case_big_sv(lib, workdir, n_reads=1000):
    pre, reads = os.path.join(workdir, "gb_sv"), os.path.join(workdir, "gb_sv.reads.fa")
    T.sim_graph(pre, 1000000, 8, 7)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 15000, "ont", 223)
    check_fasta(lib, pre + ".gfa", reads)
