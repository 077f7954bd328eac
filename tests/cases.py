"""Parity cases shared by the CPU (hostsim) and GPU (libmgb200) test modules."""
import hashlib
import os

import mgtest as T


from minigraph_b200 import capi  # noqa: E402

G = os.path.join(T.REPO, "tests", "golden")


def golden(name):
    with open(os.path.join(G, name), "rb") as f:
        return f.read()


def golden_gz(name):
    import gzip
    with gzip.open(os.path.join(G, name), "rb") as f:
        return f.read()


def case_golden_large(lib, workdir, which=("L2", "L3", "L4")):
    """the larger golden sets (tests/golden/make_golden.sh): 240 x 10 kb reads on test/MT.gfa, 240 x 15 kb on an SV graph as dense as
    the bench's MHC-scale one (1 Mb, 8 haplotypes), 200 x 20 kb HiFi-error reads with the asm preset; GAF text byte for byte"""
    if "L2" in which:
        hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mtL.reads.fa")
        T.sim_mt_haps(hap)
        T.sim_reads(hap, reads, 240, 10000, "ont", 111)
        check_gaf(lib, os.path.join(T.FIX, "MT.gfa"), reads, "lr", golden_gz("L2_MT_240x10k_ont_s111.lr.gaf.gz"))
    if "L3" in which:
        pre, reads = os.path.join(workdir, "svL"), os.path.join(workdir, "svL.reads.fa")
        T.sim_graph(pre, 1000000, 8, 7)
        T.sim_reads(pre + ".hap.fa", reads, 240, 15000, "ont", 105)
        check_gaf_lines(lib, pre + ".gfa", reads, "lr", golden("L3_sv1m_h8_s7_240x15k_ont_s105.lr.gaf.b2").split())
    if "L4" in which:
        reads = os.path.join(workdir, "mthL.reads.fa")
        T.sim_reads(os.path.join(T.FIX, "MT-human.fa"), reads, 200, 20000, "hifi", 113, circular=True)
        check_gaf(lib, os.path.join(T.FIX, "MT-human.fa"), reads, "asm", golden_gz("L4_MThuman_200x20k_hifi_s113.asm.gaf.gz"))


def first_diff(a, b):
    la, lb = a.split(b"\n"), b.split(b"\n")
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            fx, fy = x.split(b"\t"), y.split(b"\t")
            for j, (p, q) in enumerate(zip(fx, fy)):
                if p != q:
                    return "line %d field %d: %r != %r" % (i, j, p[:120], q[:120])
            return "line %d: field count %d != %d" % (i, len(fx), len(fy))
    return "line count %d != %d" % (len(la), len(lb))


def check_gaf(lib, gfa, fasta, preset, want, flag_extra=0):
    names, seqs = T.read_fasta(fasta)
    got, st = T.gaf_with_engine(lib, gfa, names, seqs, preset, flag_extra=flag_extra)
    assert got == want, first_diff(got, want)
    return st


def check_gaf_lines(lib, gfa, fasta, preset, want):
    """the GAF text against a golden file that keeps one 64-bit BLAKE2b digest (hex) per line instead of the line"""
    import hashlib
    names, seqs = T.read_fasta(fasta)
    got, st = T.gaf_with_engine(lib, gfa, names, seqs, preset)
    lines = got.split(b"\n")
    assert lines[-1] == b"", "GAF text does not end with a newline"
    assert len(lines) - 1 == len(want), "line count %d != %d" % (len(lines) - 1, len(want))
    for i, (ln, w) in enumerate(zip(lines, want)):
        assert hashlib.blake2b(ln, digest_size=8).hexdigest().encode() == w, "line %d differs from the reference's: %r" % (i, ln[:200])
    return st


def case_c1(lib, workdir):
    """config 1: test/MT.gfa <- test/MT-orangA.fa, -cx lr; md5 pinned in SURVEY.md section 8c."""
    st = check_gaf(lib, os.path.join(T.FIX, "MT.gfa"), os.path.join(T.FIX, "MT-orangA.fa"), "lr", golden("c1_MT_orangA.lr.gaf"))
    assert hashlib.md5(golden("c1_MT_orangA.lr.gaf")).hexdigest() == "22bf23ebe2039e8353f56f4a324a2eaa"
    check_gaf(lib, os.path.join(T.FIX, "MT.gfa"), os.path.join(T.FIX, "MT-chimp.fa"), "lr", golden("c1_MT_chimp.lr.gaf"))
    return st


def case_c2(lib, workdir):
    hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mt.reads.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, 24, 10000, "ont", 11)
    return check_gaf(lib, os.path.join(T.FIX, "MT.gfa"), reads, "lr", golden("c2_MT_24x10k_ont_s11.lr.gaf"))


def case_c3(lib, workdir):
    pre, reads = os.path.join(workdir, "sv"), os.path.join(workdir, "sv.reads.fa")
    T.sim_graph(pre, 300000, 3, 7)
    T.sim_reads(pre + ".hap.fa", reads, 24, 15000, "ont", 5)
    return check_gaf(lib, pre + ".gfa", reads, "lr", golden("c3_sv300k_h3_s7_24x15k_ont_s5.lr.gaf"))


def case_c4(lib, workdir):
    reads = os.path.join(workdir, "mth.reads.fa")
    T.sim_reads(os.path.join(T.FIX, "MT-human.fa"), reads, 12, 20000, "hifi", 13, circular=True)
    return check_gaf(lib, os.path.join(T.FIX, "MT-human.fa"), reads, "asm", golden("c4_MThuman_12x20k_hifi_s13.asm.gaf"))


def case_edge(lib, workdir):
    """empty, tiny, all-N, unmappable and lower-case-free reads: same objects as the reference (map-algo.c:356-360)."""
    import ctypes as C
    from minigraph_b200 import capi, options
    gfa = os.path.join(T.FIX, "MT.gfa")
    _, hs = T.read_fasta(os.path.join(T.FIX, "MT-human.fa"))
    names = [b"empty", b"tiny", b"allN", b"random", b"short_ok", b"with_N"]
    seqs = [b"", b"ACGT", b"N" * 500, (b"ACGTTGCA" * 200)[:1500], hs[0][1000:1300], hs[0][2900:3300]]
    got, _, _ = T.map_with_engine(lib, gfa, names, seqs, "lr")
    assert got[0] is None                      # qlen == 0 -> no result object
    for r in got[1:4]:
        assert r is not None and r["n_gc"] == 0
    want, _ = T.map_with_ref(gfa, names, seqs, "lr")
    for i, (a, b) in enumerate(zip(want, got)):
        assert T.diff_results(a, b) is None, (i, T.diff_results(a, b))


def case_struct_random(lib, workdir, n_reads=150, seed=23):
    """field-by-field comparison of mg_gchains_t (incl. anchors, lchains, CIGAR, ds offsets) against the reference library."""
    pre, reads = os.path.join(workdir, "svb"), os.path.join(workdir, "svb.reads.fa")
    T.sim_graph(pre, 400000, 4, 31)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 12000, "ont", seed)
    names, seqs = T.read_fasta(reads)
    want, mo_r = T.map_with_ref(pre + ".gfa", names, seqs, "lr")
    got, mo_e, st = T.map_with_engine(lib, pre + ".gfa", names, seqs, "lr")
    assert (mo_r.occ_max1, mo_r.lc_max_occ) == (mo_e.occ_max1, mo_e.lc_max_occ)
    for i, (a, b) in enumerate(zip(want, got)):
        d = T.diff_results(a, b)
        assert d is None, "read %d (%s): %s" % (i, names[i], d)
    return st


def case_wfa_fallback(lib, n_cases=12, seed=5):
    """gaps whose exact WFA exceeds the cell cap take the reference's chaining heuristic + low-memory checkpoints
    (miniwfa.c:551-601,776-834): same CIGAR and score as mwf_wfa_exact(max_iter) -> mwf_wfa_chain(step) of the reference"""
    import ctypes as C
    import random
    rng = random.Random(seed)

    def mutate(s, rate):
        out = []
        for c in s:
            u = rng.random()
            if u < rate * 0.4:
                out.append(rng.choice("ACGT"))
            elif u < rate * 0.7:
                continue
            elif u < rate:
                out.append(c)
                out.append(rng.choice("ACGT"))
            else:
                out.append(c)
        return "".join(out)
    n_fallback = 0
    for it in range(n_cases):
        n = rng.choice([300, 900, 2500])
        if it == 0:
            n = 9000  # tl + ql > 16000: beyond the 16-bit ring of tier 3, takes the 32-bit one
        t = "".join(rng.choice("ACGT") for _ in range(n))
        blocks = [mutate(t[i:i + 200], rng.choice([0.02, 0.1, 0.3]) if it else 0.02) if rng.random() < 0.8 or it == 0 else "".join(rng.choice("ACGT") for _ in range(rng.choice([50, 300])))
                  for i in range(0, n, 200)]
        q = "".join(blocks)
        ts, qs = t.encode(), q.encode()
        max_iter, step = rng.choice([(2000, 40), (20000, 25), (50000, 100), (10 ** 8, 5000)])
        if it == 0:
            max_iter, step = 10 ** 8, 5000
        gave_up, want_s, want = T.ref_wfa(ts, qs, max_iter, step)
        n_fallback += gave_up
        cap = len(ts) + len(qs) + 8
        buf = (C.c_uint32 * cap)()
        score = C.c_int(0)
        nc = lib.mgb_test_wfa(ts, len(ts), qs, len(qs), max_iter, step, buf, cap, C.byref(score))
        assert nc >= 0, (it, nc)
        got = [buf[i] for i in range(nc)]
        assert got == want and score.value == want_s, "case %d (tl=%d ql=%d max_iter=%d step=%d): score %d vs %d" % (it, len(ts), len(qs), max_iter, step, score.value, want_s)
    assert n_fallback >= 3


def check_cigar_invariants(r, qlen):
    """what holds for every mg_gchains_t the reference produces with -c (checked against the reference itself in
    test_hostsim_parity.py): the CIGAR of a chain spans exactly its query and path intervals and sums to its mlen/blen"""
    for g in r["gc"]:
        assert 0 <= g["qs"] < g["qe"] <= qlen and 0 <= g["ps"] < g["pe"] <= g["plen"], g
        if g["cigar"] is None:
            continue
        n_cigar, mlen, blen, aplen, ss, ee = g["cigar_hdr"]
        assert n_cigar == len(g["cigar"]) and all((c & 15) in (1, 2, 7, 8) and (c >> 4) > 0 for c in g["cigar"])
        assert sum(c >> 4 for c in g["cigar"] if (c & 15) in (7, 8, 1)) == g["qe"] - g["qs"]
        assert sum(c >> 4 for c in g["cigar"] if (c & 15) in (7, 8, 2)) == g["pe"] - g["ps"] == aplen
        assert sum(c >> 4 for c in g["cigar"] if (c & 15) == 7) == mlen and sum(c >> 4 for c in g["cigar"]) == blen
        assert all((a & 15) != (b & 15) for a, b in zip(g["cigar"], g["cigar"][1:]))  # adjacent operations are merged


def case_full_size(lib, workdir, n_reads=10000, n_sub=300, n_ref=100, seed=11):
    """BASELINE config 2 at its full size (10 000 x 10 kb ONT-like reads on test/MT.gfa), through properties that do not
    need the reference on every read: (1) reads sampled from the graph map (all but a stray one) and a CIGAR is
    consistent with its intervals; (2) a result does not depend on the batch a read travels in (mg_map_frag is a pure function of the read,
    map-algo.c:340-495): a shuffled sample mapped as its own batch gives the same objects; (3) a smaller sample against
    the reference library itself."""
    import ctypes as C
    import random
    from minigraph_b200 import capi, options
    hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mt.full.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, n_reads, 10000, "ont", seed)
    names, seqs = T.read_fasta(reads)
    n = len(seqs)
    assert n == n_reads
    gfa = os.path.join(T.FIX, "MT.gfa")
    g = lib.mgb_gfa_read(gfa.encode())
    io, mo = options.opt_set("lr", True)
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()
    qlens = (C.c_int * n)(*[len(s) for s in seqs])
    cseqs, cnames = (C.c_char_p * n)(*seqs), (C.c_char_p * n)(*names)
    gcs = (C.POINTER(capi.mg_gchains_t) * n)()
    assert lib.mg_map_batch(gi, n, qlens, cseqs, cnames, gcs, C.byref(mo)) == 0, lib.mgb_last_error()
    n_mapped = sum(1 for i in range(n) if gcs[i] and gcs[i].contents.n_gc > 0)
    assert n_mapped >= 0.999 * n, "%d of %d reads sampled from the graph did not map" % (n - n_mapped, n)
    rng = random.Random(seed)
    sub = rng.sample(range(n), min(n_sub, n))
    full = {i: T.gchains_to_py(gcs[i]) for i in sub}
    lib.mgb_free_batch(n, gcs)
    for i in sub:
        check_cigar_invariants(full[i], len(seqs[i]))
    m = len(sub)
    qlens2 = (C.c_int * m)(*[len(seqs[i]) for i in sub])
    cseqs2, cnames2 = (C.c_char_p * m)(*[seqs[i] for i in sub]), (C.c_char_p * m)(*[names[i] for i in sub])
    gcs2 = (C.POINTER(capi.mg_gchains_t) * m)()
    assert lib.mg_map_batch(gi, m, qlens2, cseqs2, cnames2, gcs2, C.byref(mo)) == 0, lib.mgb_last_error()
    for j, i in enumerate(sub):
        d = T.diff_results(T.gchains_to_py(gcs2[j]), full[i])
        assert d is None, "read %d: alone vs in the full batch: %s" % (i, d)
    lib.mgb_free_batch(m, gcs2)
    lib.mg_idx_destroy(gi)
    lib.mgb_gfa_destroy(g)
    if n_ref > 0:
        pick = sub[:n_ref]
        want, _ = T.map_with_ref(gfa, [names[i] for i in pick], [seqs[i] for i in pick], "lr")
        for i, w in zip(pick, want):
            if not isinstance(w, T.Digest):  # a stored result is known by its digest only
                check_cigar_invariants(w, len(seqs[i]))  # the invariants are the reference's, not ours
            d = T.diff_results(full[i], w)
            assert d is None, "read %d vs reference: %s" % (i, d)


def case_wfa_divergent(lib, n_cases=24, seed=5):
    """unrelated sequences of unequal length: the band reaches the matrix borders, is re-centred and shrinks
    (miniwfa.c:144-171) -- what the tier-3 ring has to get right when slots are reused by narrower wavefronts"""
    import ctypes as C
    import random
    rng = random.Random(seed)
    for it in range(n_cases):
        tl = rng.choice([150, 300, 500, 800])
        ql = max(20, int(tl * rng.choice([0.3, 0.7, 1.0, 1.5])))
        t = "".join(rng.choice("ACGT") for _ in range(tl))
        q = "".join(rng.choice("ACGT") for _ in range(ql))
        if it % 3 == 0:  # a shared core between random flanks
            core = "".join(rng.choice("ACGT") for _ in range(100))
            t, q = t[:tl // 2] + core + t[tl // 2:], q[:ql // 3] + core + q[ql // 3:]
        ts, qs = t.encode(), q.encode()
        _, want_s, want = T.ref_wfa(ts, qs, 10 ** 8)
        assert want_s >= 0
        cap = len(ts) + len(qs) + 8
        buf = (C.c_uint32 * cap)()
        score = C.c_int(0)
        nc = lib.mgb_test_wfa(ts, len(ts), qs, len(qs), 10 ** 8, 5000, buf, cap, C.byref(score))
        assert nc >= 0 and [buf[i] for i in range(nc)] == want and score.value == want_s, (it, tl, ql, score.value, want_s)


def case_wfa_band_shrinks(lib, n_cases=48, seed=99):
    """tier 3 far past score 256: unrelated pairs, noisy copies with a long indel, shared cores between random flanks, low-complexity
    pairs.  The ring keeps 17 H slots but only 3 / 2 slots of E/F; what the band shrink (miniwfa.c:144-171) wants to know about the
    last 17 wavefronts comes from the last-good-score slice.  Same CIGAR and score as the reference's mwf_wfa_exact()."""
    import ctypes as C
    import random
    rng = random.Random(seed)
    n_shrunk = 0
    for it in range(n_cases):
        tl = rng.choice([200, 400, 700, 1200, 2000])
        ql = max(30, int(tl * rng.choice([0.2, 0.5, 0.8, 1.0, 1.3, 2.0])))
        t = "".join(rng.choice("ACGT") for _ in range(tl))
        mode = it % 4
        if mode == 0:
            q = "".join(rng.choice("ACGT") for _ in range(ql))
        elif mode == 1:
            q = "".join(c if rng.random() > 0.25 else rng.choice("ACGT") for c in t)
            cut = rng.randrange(len(q))
            q = q[:cut] + q[cut + rng.choice([50, 150, 400]):]
        elif mode == 2:
            q = "".join(rng.choice("ACGT") for _ in range(ql))
            for _ in range(3):
                core = "".join(rng.choice("ACGT") for _ in range(rng.choice([30, 80])))
                i, j = rng.randrange(len(t)), rng.randrange(len(q))
                t, q = t[:i] + core + t[i:], q[:j] + core + q[j:]
        else:
            q = "".join(rng.choice("AC") for _ in range(ql))
            t = "".join(rng.choice("AC") if rng.random() < 0.7 else rng.choice("GT") for _ in range(tl))
        if not q:
            continue
        ts, qs = t.encode(), q.encode()
        _, want_s, want = T.ref_wfa(ts, qs, 10 ** 8)
        assert want_s >= 0
        n_shrunk += want_s >= 256
        cap = len(ts) + len(qs) + 8
        buf = (C.c_uint32 * cap)()
        score = C.c_int(0)
        nc = lib.mgb_test_wfa(ts, len(ts), qs, len(qs), 10 ** 8, 5000, buf, cap, C.byref(score))
        assert nc >= 0 and [buf[i] for i in range(nc)] == want and score.value == want_s, (it, len(ts), len(qs), score.value, want_s, nc)
    assert n_shrunk >= n_cases // 2


def case_radix_exact(lib, n_cases=60, seed=17):
    """the warp-wide replay of klib's unstable radix sort (mgb_common.cuh radix_sort_exact_w), in place and as a walk over digits, with
    scratch on "chip" and in the arena: the same order as radix_sort_128x() of the reference, ties included (ksort.h:112-162) --
    few distinct keys (long runs of ties), keys that differ in one byte only (one level), bins above 64 elements (recursion), skewed bins"""
    import ctypes as C
    import random
    from minigraph_b200 import capi
    lib.mgb_test_radix128.restype = C.c_int
    lib.mgb_test_radix128.argtypes = [C.POINTER(capi.mg128_t), C.c_int64, C.c_int, C.c_int]
    rng = random.Random(seed)
    for it in range(n_cases):
        n = rng.choice([65, 191, 192, 193, 700, 1100, 3000, 9000])
        nk = rng.choice([2, 7, 300, 5000, 2 ** 40])
        sh = rng.choice([0, 8, 16, 33])
        base = rng.randrange(2 ** 20) << 40
        if it % 5 == 4:  # one heavy bin and a sprinkle of others
            keys = [base + ((rng.randrange(nk) << sh) if rng.random() < 0.1 else (3 << sh)) for _ in range(n)]
        else:
            keys = [base + (rng.randrange(nk) << sh) for _ in range(n)]
        want = T.ref_radix_sort([(x, i) for i, x in enumerate(keys)])
        for walk, hot in ((0, 0), (1, 0), (1, 16384), (1, n // 4 + 3400), (0, 16384)):  # (n/4 + 3400: what the callers ask of the on-chip slice; the digits then go to the arena)
            got = (capi.mg128_t * n)()
            for i, x in enumerate(keys):
                got[i].x, got[i].y = x, i
            rc = lib.mgb_test_radix128(got, n, walk, hot)
            assert rc == 0, (it, n, walk, hot, rc)
            gl = [(got[i].x, got[i].y) for i in range(n)]
            if isinstance(want, T.Digest):
                assert gl == want, "case %d (n=%d, %d keys << %d, walk=%d, hot=%d): not the reference's order" % (it, n, nk, sh, walk, hot)
                continue
            bad = next((i for i in range(n) if gl[i] != want[i]), None)
            assert bad is None, "case %d (n=%d, %d keys << %d, walk=%d, hot=%d): position %d holds element %d, the reference has %d" % (
                it, n, nk, sh, walk, hot, bad, gl[bad][1], want[bad][1])


def case_wfa_tiers(lib, workdir, n_struct=60):
    """the gap alignment tiers (mgb_wfa_tiers.cuh: slices that hold -inf outside their range instead of bounds checks).  Same GAF
    for the golden cases (lr and asm presets, both on-chip tiers busy), same mg_gchains_t fields as the reference on an SV graph,
    also with the learned tier routing of a second batch"""
    from minigraph_b200 import capi
    for fn in (case_c2, case_c3, case_c4):
        st = fn(lib, workdir)
        prof = {n: st.prof[i] for i, n in enumerate(capi.PROF_NAMES)}
        assert prof["wfa_fast_n"] > 500, prof
        assert fn is case_c4 or prof["wfa_mid_n"] > 500, prof
    case_struct_random(lib, workdir, n_reads=n_struct, seed=37)
    case_tier_routing(lib, workdir)
    case_short_reads(lib, workdir, n_pairs=20)  # sr preset: tier 1 only, two-segment fragments
    case_wfa_fallback(lib)  # tier 3 against miniwfa: scores far past 256 (band re-centring), capped runs, a gap beyond the 16-bit ring
    case_wfa_divergent(lib)
    case_wfa_band_shrinks(lib)


def case_gchain_labels(lib, workdir, n_reads=150, graph_len=1000000):
    """graph chaining from the per-source label table (mgb_gclabel.cuh) on a graph dense enough that every read spans a dozen
    segments: every field against the reference with the table on (sources searched once per batch by k_gc_labels), with the
    table off (every read searches its own sources), lr and asm presets (walk bounds of 20 kb and 150 kb)"""
    pre, reads = os.path.join(workdir, "svl"), os.path.join(workdir, "svl.reads.fa")
    T.sim_graph(pre, graph_len, 8, 7)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 15000, "ont", 5)
    names, seqs = T.read_fasta(reads)
    try:
        for preset, m in (("lr", n_reads), ("asm", n_reads // 3)):
            want, _ = T.map_with_ref(pre + ".gfa", names[:m], seqs[:m], preset)
            for cache in (1, 0):
                assert lib.mgb_set_param(b"lab_cache", cache) == 0
                got, _, st = T.map_with_engine(lib, pre + ".gfa", names[:m], seqs[:m], preset)
                assert (st.n_lab_new > 100) == bool(cache), (preset, cache, st.n_lab_new)
                assert sum(r["n_lc"] for r in got if r) > 5 * m  # the reads do span many segments
                for i, (a, b) in enumerate(zip(want, got)):
                    d = T.diff_results(a, b)
                    assert d is None, "%s lab_cache=%d read %d: %s" % (preset, cache, i, d)
    finally:
        lib.mgb_set_param(b"lab_cache", 1)


def case_tandem_diagonals(lib, workdir, n_reads=48, seed=29):
    """RMQ chaining where two diagonals interleave in target order: a linear reference with tandem duplications (copies 700 bp and
    3 kb apart: narrow and wide blocks of the outer query's summaries, mgb_lchain.cuh chain_rmq_fill_w) and a circular one whose reads
    wrap around; asm preset (RMQ chaining of every read) and lr (the long-join rescue); every field against the reference"""
    import random
    rng = random.Random(seed)

    def rnd(n):
        return "".join(rng.choice("ACGT") for _ in range(n))
    d1, d2 = rnd(700), rnd(3000)
    ref = rnd(6000) + d1 + d1 + d1 + rnd(5000) + d2 + d2 + rnd(7000) + d1 + rnd(4000)
    lin = os.path.join(workdir, "tandem.fa")
    with open(lin, "w") as f:
        f.write(">tandem\n%s\n" % ref)
    for gfa, circular, tag in ((lin, False, "lin"), (os.path.join(T.FIX, "MT-human.fa"), True, "circ")):
        for preset, err, rl in (("asm", "hifi", 18000), ("lr", "ont", 11000)):
            reads = os.path.join(workdir, "tandem.%s.%s.fa" % (tag, preset))
            T.sim_reads(gfa, reads, n_reads, rl, err, seed + len(tag) + len(preset), circular=circular)
            names, seqs = T.read_fasta(reads)
            want, _ = T.map_with_ref(gfa, names, seqs, preset)
            got, _, _ = T.map_with_engine(lib, gfa, names, seqs, preset)
            assert sum(1 for r in want if r and r["n_gc"] > 0) >= n_reads // 2, (tag, preset)
            for i, (a, b) in enumerate(zip(want, got)):
                d = T.diff_results(a, b)
                assert d is None, "%s %s read %d: %s" % (tag, preset, i, d)


def case_chain_skip(lib, workdir, n_reads=40):
    """max_lc_skip far below its default (25): the early stop of the chaining DP and of the RMQ walk -- "too many candidates in
    a row that are already on a better chain" (lchain.c:185-190, 336-343) -- fires all the time instead of almost never;
    every field against the reference, DP chaining (lr) and RMQ chaining (asm)"""
    pre, reads = os.path.join(workdir, "svc"), os.path.join(workdir, "svc.reads.fa")
    T.sim_graph(pre, 300000, 3, 19)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 12000, "ont", 47)
    names, seqs = T.read_fasta(reads)
    for preset in ("lr", "asm"):
        for skip in (1, 3):
            def tweak(mo, skip=skip):
                mo.max_lc_skip = skip
            want, _ = T.map_with_ref(pre + ".gfa", names, seqs, preset, tweak=tweak)
            got, _, _ = T.map_with_engine(lib, pre + ".gfa", names, seqs, preset, tweak=tweak)
            for i, (a, b) in enumerate(zip(want, got)):
                d = T.diff_results(a, b)
                assert d is None, "%s max_lc_skip=%d read %d: %s" % (preset, skip, i, d)


def case_switches(lib, workdir, device):
    """the engine's experiment switches change the schedule, never the result: the same golden GAF with each of them on"""
    settings = [{b"lab_cache": 0}]  # graph chaining without the label table
    if device:
        settings += [{b"sw8": 1, b"mb8": 16, b"sw7": 1, b"mb7": 16}]  # one-warp blocks for the tail-bound job kernels
    defaults = {b"lab_cache": 1, b"sw8": 4, b"mb8": 4, b"sw7": 4, b"mb7": 4}
    for st in settings:
        try:
            for k, v in st.items():
                assert lib.mgb_set_param(k, v) == 0
            case_c3(lib, workdir)
        finally:
            for k in st:
                lib.mgb_set_param(k, defaults[k])


def case_concurrent_calls(lib, workdir, n_threads=3, n_reads=90):
    """mg_map_batch() entered by several host threads at once on one index (each call takes a slot of its own; the reference's
    mg_map is re-entrant per thread buffer, minigraph.h:167-170): every thread gets what a single caller gets"""
    import ctypes as C
    import threading
    from minigraph_b200 import capi, options
    pre, reads = os.path.join(workdir, "svt"), os.path.join(workdir, "svt.reads.fa")
    T.sim_graph(pre, 400000, 4, 23)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 9000, "ont", 61)
    names, seqs = T.read_fasta(reads)
    g = lib.mgb_gfa_read((pre + ".gfa").encode())
    io, mo = options.opt_set("lr", True)
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()

    def run(lo, hi, out):
        n = hi - lo
        qlens = (C.c_int * n)(*[len(x) for x in seqs[lo:hi]])
        cs, cn = (C.c_char_p * n)(*seqs[lo:hi]), (C.c_char_p * n)(*names[lo:hi])
        gcs = (C.POINTER(capi.mg_gchains_t) * n)()
        rc = lib.mg_map_batch(gi, n, qlens, cs, cn, gcs, C.byref(mo))
        out.append((lo, rc, [T.gchains_to_py(gcs[i]) for i in range(n)]))
        lib.mgb_free_batch(n, gcs)

    whole = []
    run(0, n_reads, whole)
    assert whole[0][1] == 0
    for rnd in range(2):  # the second round finds the label table warm
        parts, th = [], []
        for t in range(n_threads):
            th.append(threading.Thread(target=run, args=(n_reads * t // n_threads, n_reads * (t + 1) // n_threads, parts)))
        for x in th:
            x.start()
        for x in th:
            x.join()
        assert len(parts) == n_threads
        for lo, rc, res in parts:
            assert rc == 0, lib.mgb_last_error()
            for i, r in enumerate(res):
                d = T.diff_results(whole[0][2][lo + i], r)
                assert d is None, "round %d read %d: %s" % (rnd, lo + i, d)
    lib.mg_idx_destroy(gi)
    lib.mgb_gfa_destroy(g)


def case_index_big(lib, workdir, graph_len=50000000, n_probe=40000):
    """the minimizer table of a graph whose index does not fit L2 (built on the device, mgb_index.cuh) against the reference's
    (index.c:115-165): the same occurrence list -- content and order -- for tens of thousands of probed minimizers and for keys
    that are not there, the same quantile-derived mapping options (options.c:120-134), and the switch back to the host build"""
    import ctypes as C
    import random
    from minigraph_b200 import options
    pre = os.path.join(workdir, "big")
    T.sim_graph(pre, graph_len, 3, 17)
    with open(pre + ".gfa") as f:  # repeats: sixty segments once more under another name, so that many minimizers have occurrence lists
        dup = [ln.split("\t") for ln in f if ln.startswith("S\t")][100:160]
    with open(pre + ".gfa", "a") as f:
        for i, t in enumerate(dup):
            f.write("\t".join([t[0], "dup%d" % i] + t[2:]))
    # probes: the minimizers of random stretches of the graph (through the oracle's sketch, which is the reference's: test_oracle.py),
    # plus random keys
    orc = T.load_oracle()
    io, _ = options.opt_set("lr")
    g = lib.mgb_gfa_read((pre + ".gfa").encode())
    rnd = random.Random(5)
    keys = set()
    n_seg = g.contents.n_seg
    while len(keys) < n_probe:
        seg = g.contents.seg[rnd.randrange(n_seg) if len(keys) % 4 else n_seg - 1 - rnd.randrange(60)]
        if seg.len < 200:
            continue
        st = rnd.randrange(seg.len - 199)
        for x, _ in T.orc_sketch(orc, C.string_at(seg.seq, seg.len)[st:st + 200], io.w, io.k, 0):
            keys.add(x >> 8)
    lib.mgb_gfa_destroy(g)
    keys = sorted(keys) + [rnd.getrandbits(2 * io.k) for _ in range(2000)]

    def compute():
        ref = T.load_ref()
        rg = ref.gfa_read((pre + ".gfa").encode())
        io_r, rmo = options.opt_set("lr")
        rgi = ref.mg_index(rg, C.byref(io_r), 8, C.byref(rmo))
        assert rgi
        n1 = C.c_int(0)
        lists = []
        for k in keys:
            a = ref.mg_idx_get(rgi, k, C.byref(n1))
            lists.append([a[i] for i in range(n1.value)])
        ref.mg_idx_destroy(rgi)
        ref.gfa_destroy(rg)
        return [rmo.occ_max1, rmo.lc_max_occ, rmo.bw_long], lists, sum(len(x) > 1 for x in lists)
    want_mo, want, n_multi = T.reference("mg_idx_get", (T.file_digest(pre + ".gfa"), bytes(io), T.digest(keys)), compute,
                                         lambda v: [v[0], T.digest(v[1]), v[2]], lambda s: (s[0], T.Digest(s[1]), s[2]))
    assert n_multi > 100, n_multi
    n2 = C.c_int(0)
    for index_dev in (1, 0):
        assert lib.mgb_set_param(b"index_dev", index_dev) == 0
        try:
            g = lib.mgb_gfa_read((pre + ".gfa").encode())
            io2, mo = options.opt_set("lr")
            gi = lib.mg_index(g, C.byref(io2), 1, C.byref(mo))
            assert gi, lib.mgb_last_error()
            assert [mo.occ_max1, mo.lc_max_occ, mo.bw_long] == want_mo
            got = []
            for k in keys:
                b = lib.mg_idx_get(gi, k, C.byref(n2))
                got.append([b[i] for i in range(n2.value)])
            if isinstance(want, T.Digest):
                assert got == want, "index_dev=%d: the occurrence lists of the probed keys are not the reference's" % index_dev
            for k, x, y in zip(keys, got, [] if isinstance(want, T.Digest) else want):
                assert x == y, (hex(k), len(x), len(y))
            lib.mg_idx_destroy(gi)
            lib.mgb_gfa_destroy(g)
        finally:
            lib.mgb_set_param(b"index_dev", 1)


def case_multi_device(lib, workdir, devices="0,0,0", n_reads=100):
    """MGB_DEVICES: the index replicated on several devices (here the same one three times, which runs the same code), every
    mg_map_batch() cut into one contiguous part per device: the results, in input order, are what one device gives"""
    pre, reads = os.path.join(workdir, "svm"), os.path.join(workdir, "svm.reads.fa")
    T.sim_graph(pre, 300000, 3, 31)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 7000, "ont", 71)
    names, seqs = T.read_fasta(reads)
    one, _, _ = T.map_with_engine(lib, pre + ".gfa", names, seqs, "lr")
    os.environ["MGB_DEVICES"] = devices
    try:
        many, _, _ = T.map_with_engine(lib, pre + ".gfa", names, seqs, "lr")
    finally:
        del os.environ["MGB_DEVICES"]
    assert sum(1 for r in one if r and r["n_gc"] > 0) > n_reads // 2
    for i, (a, b) in enumerate(zip(one, many)):
        d = T.diff_results(a, b)
        assert d is None, "read %d: %s" % (i, d)


def case_upload_modes(lib, workdir, n_reads=80):
    """how the reads reach the device does not change what comes back: 2 bits per base (all A/C/G/T), the same with a few reads that
    hold N or lower-case letters (those travel as ASCII beside the packed ones), the whole batch as ASCII (many such reads), and the
    pack2=0 switch; every field against the reference, whose alignment compares raw bytes (N matches N, 'a' does not match 'A')"""
    pre, reads = os.path.join(workdir, "svu"), os.path.join(workdir, "svu.reads.fa")
    T.sim_graph(pre, 300000, 3, 29)
    T.sim_reads(pre + ".hap.fa", reads, n_reads, 6000, "ont", 67)
    names, seqs = T.read_fasta(reads)

    def spoil(s, k):
        b = bytearray(s)
        b[1000 + k] = ord("N")
        b[3000:3004] = b[3000:3004].lower()
        return bytes(b)
    few = [spoil(s, i) if i % 29 == 0 else s for i, s in enumerate(seqs)]
    many = [spoil(s, i) for i, s in enumerate(seqs)]
    try:
        for tag, ss, pack in (("packed", seqs, 1), ("few", few, 1), ("many", many, 1), ("switch", seqs, 0)):
            assert lib.mgb_set_param(b"pack2", pack) == 0
            want, _ = T.map_with_ref(pre + ".gfa", names, ss, "lr")
            got, _, st = T.map_with_engine(lib, pre + ".gfa", names, ss, "lr")
            bases = sum(len(x) for x in ss)
            assert (st.h2d_bytes < bases // 2) == (tag in ("packed", "few")), (tag, st.h2d_bytes, bases)
            for i, (a, b) in enumerate(zip(want, got)):
                d = T.diff_results(a, b)
                assert d is None, "%s read %d: %s" % (tag, i, d)
    finally:
        lib.mgb_set_param(b"pack2", 1)


def case_tier_routing(lib, workdir, n_reads=120):
    """the WFA tier thresholds learned from one batch route the gaps of the next: same results, and the routing did engage"""
    import ctypes as C
    from minigraph_b200 import capi, options
    hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mt.route.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, n_reads, 10000, "ont", 29)
    names, seqs = T.read_fasta(reads)
    g = lib.mgb_gfa_read(os.path.join(T.FIX, "MT.gfa").encode())
    io, mo = options.opt_set("lr", True)
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()
    n = len(seqs)
    qlens = (C.c_int * n)(*[len(s) for s in seqs])
    cseqs, cnames = (C.c_char_p * n)(*seqs), (C.c_char_p * n)(*names)
    runs, st = [], capi.mgb_stats_t()
    for it in range(2):
        gcs = (C.POINTER(capi.mg_gchains_t) * n)()
        assert lib.mg_map_batch(gi, n, qlens, cseqs, cnames, gcs, C.byref(mo)) == 0, lib.mgb_last_error()
        runs.append([T.gchains_to_py(gcs[i]) for i in range(n)])
        lib.mgb_free_batch(n, gcs)
        lib.mgb_get_stats(gi, C.byref(st))
        if it == 0:
            assert st.skip1_len > 1 << 30  # nothing learned yet: every gap tries every tier
    assert st.skip1_len < 400 and st.skip2_len >= st.skip1_len, (st.skip1_len, st.skip2_len)
    for i, (a, b) in enumerate(zip(*runs)):
        d = T.diff_results(a, b)
        assert d is None, "read %d differs between the unrouted and the routed batch: %s" % (i, d)
    lib.mg_idx_destroy(gi)


def case_multi_segment(lib, workdir, n_frag=40):
    """fragments of 2-3 segments through mg_map_frag (paired reads): one result for the concatenated fragment, no CIGAR, same
    fields as the reference (map-algo.c:34-45,356-360,402,407,464,475)"""
    import ctypes as C
    import random
    from minigraph_b200 import options
    hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mt.seg.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, n_frag, 9000, "ont", 53)
    names, seqs = T.read_fasta(reads)
    rng = random.Random(7)
    frags = []
    for nm, s in zip(names, seqs):
        n_seg = rng.choice([2, 2, 3])
        cut = sorted(rng.sample(range(1500, len(s) - 1500), n_seg - 1))
        parts = [s[a:b] for a, b in zip([0] + cut, cut + [len(s)])]
        if rng.random() < 0.3:
            parts[-1] = parts[-1][:40]  # a segment too short to be sketched in chunks
        frags.append((nm, parts))
    gfa = os.path.join(T.FIX, "MT.gfa")
    want = T.map_frag_with_ref(gfa, frags, "lr", True)
    io, mo = options.opt_set("lr", True)
    g = lib.mgb_gfa_read(gfa.encode())
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()
    got = map_frags(lib, gi, mo, frags)
    lib.mg_idx_destroy(gi)
    n_mapped = 0
    for (nm, parts), w, r in zip(frags, want, got):
        d = T.diff_results(w, r)
        assert d is None, (nm, [len(x) for x in parts], d)
        if w and w["n_gc"] > 0:
            n_mapped += 1
    assert n_mapped >= n_frag // 2


def map_frags(lib, gi, mo, frags):
    """mg_map_frag() of an engine library on every fragment (name, [segment sequences]), one call each"""
    import ctypes as C
    b = lib.mg_tbuf_init()
    lib.mg_map_frag.restype = None
    lib.mg_map_frag.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.POINTER(capi.mg_gchains_t)), C.c_void_p, C.c_void_p, C.c_char_p]
    res = []
    for nm, parts in frags:
        n_seg = len(parts)
        gcs = (C.POINTER(capi.mg_gchains_t) * n_seg)()
        lib.mg_map_frag(C.cast(gi, C.c_void_p), n_seg, (C.c_int * n_seg)(*[len(x) for x in parts]), (C.c_char_p * n_seg)(*parts), gcs, b,
                        C.cast(C.pointer(mo), C.c_void_p), nm)
        assert all(not gcs[i] for i in range(1, n_seg))
        res.append(T.gchains_to_py(gcs[0]))
        lib.mg_gchain_free(gcs[0])
    lib.mg_tbuf_destroy(b)
    return res


def case_short_reads(lib, workdir, n_pairs=60):
    """the `sr` preset: seeds by heap merge instead of the radix sort (map-algo.c:93-150), short-read chaining gaps, read
    pairs as two-segment fragments -- every field against the reference's mg_map_frag"""
    import ctypes as C
    import random
    from minigraph_b200 import capi, options
    hap, reads = os.path.join(workdir, "mt.hap.fa"), os.path.join(workdir, "mt.sr.fa")
    T.sim_mt_haps(hap)
    T.sim_reads(hap, reads, n_pairs, 500, "hifi", 61)
    names, seqs = T.read_fasta(reads)
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    rng = random.Random(3)
    gfa = os.path.join(T.FIX, "MT.gfa")
    frags = []
    for nm, s in zip(names, seqs):
        if rng.random() < 0.7:  # a pair: 150 bases from each end, the mate reverse-complemented
            parts = [s[:150], s[-150:].translate(comp)[::-1]]
        else:
            parts = [s[:rng.choice([100, 150, 250])]]
        frags.append((nm, parts))
    want = T.map_frag_with_ref(gfa, frags, "sr", False)
    io, mo = options.opt_set("sr", False)
    g_e = lib.mgb_gfa_read(gfa.encode())
    gi_e = lib.mg_index(g_e, C.byref(io), 1, C.byref(mo))
    assert gi_e, lib.mgb_last_error()
    got = map_frags(lib, gi_e, mo, frags)
    n_mapped = 0
    for (nm, parts), w, r in zip(frags, want, got):
        d = T.diff_results(w, r)
        assert d is None, (nm, [len(x) for x in parts], d)
        if w and w["n_gc"] > 0:
            n_mapped += 1
    assert n_mapped >= n_pairs // 2, n_mapped
    # the same fragments in one call of the batch entry point
    flat = [x for _, parts in frags for x in parts]
    n_tot = len(flat)
    nseg = (C.c_int * len(frags))(*[len(parts) for _, parts in frags])
    ql = (C.c_int * n_tot)(*[len(x) for x in flat])
    sq = (C.c_char_p * n_tot)(*flat)
    nms = (C.c_char_p * len(frags))(*[nm for nm, _ in frags])
    gcs = (C.POINTER(capi.mg_gchains_t) * n_tot)()
    assert lib.mg_map_batch_frag(gi_e, len(frags), nseg, ql, sq, nms, gcs, C.byref(mo)) == 0, lib.mgb_last_error()
    off = 0
    for f, (nm, parts) in enumerate(frags):
        assert all(not gcs[off + j] for j in range(1, len(parts)))
        d = T.diff_results(want[f], T.gchains_to_py(gcs[off]))
        assert d is None, (nm, d)
        off += len(parts)
    lib.mgb_free_batch(n_tot, gcs)
    lib.mg_idx_destroy(gi_e)


def case_no_diag(lib, workdir):
    """MG_M_NO_DIAG (-D): a read that carries the name of the sequence it comes from loses the seeds on its own diagonal
    (map-algo.c:167-178): same result fields as the reference, for a full self copy, a prefix, an inner piece and a stranger"""
    fa = os.path.join(T.FIX, "MT-human.fa")
    gname, hs = T.read_fasta(fa)
    full = hs[0]
    names = [gname[0], gname[0], gname[0], b"someone_else", gname[0] + b"x"]
    seqs = [full, full[:6000], full[3000:9000], full[:6000], full[:6000]]
    import minigraph_b200.options as options_mod
    orig = options_mod.opt_set

    def with_flag(preset=None, cigar=True):
        io, mo = orig(preset, cigar)
        mo.flag |= 0x400000  # MG_M_NO_DIAG (minigraph.h:27)
        return io, mo
    options_mod.opt_set = with_flag
    T.options.opt_set = with_flag
    try:
        got, _, _ = T.map_with_engine(lib, fa, names, seqs, "asm")
        want, _ = T.map_with_ref(fa, names, seqs, "asm")
    finally:
        options_mod.opt_set = orig
        T.options.opt_set = orig
    for i, (a, b) in enumerate(zip(want, got)):
        d = T.diff_results(a, b)
        assert d is None, (i, d)
    plain, _ = T.map_with_ref(fa, names[:2], seqs[:2], "asm")
    assert T.diff_results(plain[1], want[1]) is not None  # the flag did change something for the self-named prefix
