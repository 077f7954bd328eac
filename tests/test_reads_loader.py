"""mgb_reads_load(): the library's own FASTA/FASTQ reader (input side, SURVEY 8f-3) against the reference's bseq.c on the same files."""
import ctypes as C
import gzip
import os

import mgtest as T
from minigraph_b200 import capi


def load(lib, fn, max_bases=0):
    r = lib.mgb_reads_load(fn.encode(), max_bases)
    assert r
    c = r.contents
    out = [(c.name[i], C.string_at(c.seq[i], c.len[i])) for i in range(c.n_reads)]
    assert c.n_bases == sum(len(s) for _, s in out)
    lib.mgb_reads_free(r)
    return out


def ref_load(fn):
    """the reference's reader: mg_bseq_open / mg_bseq_read (bseq.c:31-98), sequences as it hands them to the mapper (before gmap.c:81 upper-casing)"""
    def compute():
        ref = T.load_ref()

        class bseq1(C.Structure):
            _fields_ = [("l_seq", C.c_int), ("rid", C.c_int), ("name", C.c_char_p), ("seq", C.c_void_p), ("qual", C.c_void_p), ("comment", C.c_void_p)]
        ref.mg_bseq_open.restype = C.c_void_p
        ref.mg_bseq_read.restype = C.POINTER(bseq1)
        ref.mg_bseq_read.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        ref.mg_bseq_close.argtypes = [C.c_void_p]
        fp = ref.mg_bseq_open(fn.encode())
        assert fp
        n = C.c_int(0)
        out = []
        while True:
            s = ref.mg_bseq_read(fp, 1 << 30, 0, 0, 0, C.byref(n))
            if n.value == 0:
                break
            out += [(s[i].name, C.string_at(s[i].seq, s[i].l_seq).upper()) for i in range(n.value)]
        ref.mg_bseq_close(fp)
        return out
    # a gzip file is keyed by what it holds: its bytes carry the time it was written
    with (gzip.open if fn.endswith(".gz") else open)(fn, "rb") as f:
        key = T.digest(f.read())
    return T.reference("mg_bseq_read", (key,), compute, T.digest, T.Digest)


def test_reader_matches_bseq(tmp_path):
    lib = T.load_hostsim()
    capi.bind_engine_api(lib)
    fa = str(tmp_path / "a.fa")
    with open(fa, "w") as f:
        f.write(">r1 comment here\nACGTacgtNN\nGGGG\n\n>r2\tx\nTTTT\r\n>r3\n>r4 empty before\nAC\n")
    fq = str(tmp_path / "b.fq.gz")
    with gzip.open(fq, "wt") as f:
        f.write("@q1 c\nACGTAC\nGT\n+\n@@@@>>II\n@q2\nacgtn\n+q2\n>>>@@\n")
    for fn in (fa, fq, os.path.join(T.FIX, "MT-chimp.fa")):
        got, want = load(lib, fn), ref_load(fn)
        assert got == want, (fn, got[:3], str(want)[:300])
    assert len(load(lib, fa, max_bases=15)) == 2  # stops after the record that reaches the limit
    assert not lib.mgb_reads_load(b"/nonexistent/file.fa", 0)
