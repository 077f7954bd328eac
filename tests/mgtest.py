"""Shared helpers of the test-suite: oracle bindings, FASTA reader, deep comparison of mg_gchains_t objects, and the
stored results of the reference (tests/golden/reference_results.json) that stand in for it where it is not built."""
import atexit
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from minigraph_b200 import capi  # noqa: E402
from minigraph_b200 import options  # noqa: E402

FIX = os.path.join(REPO, "tests", "golden", "fixtures")
REF_SO = os.path.join(REPO, "oracle", "_ref", "libmgref.so")
REF_BIN = os.path.join(REPO, "oracle", "_ref", "minigraph")
HOSTSIM_SO = os.path.join(REPO, "tests", "hostsim", "libmgb_hostsim.so")
MGSIM = os.path.join(REPO, "tools", "mgsim")
REF_STORE = os.path.join(REPO, "tests", "golden", "reference_results.json")


def have_ref():
    return os.path.exists(REF_SO) and os.path.exists(REF_BIN)


def digest(obj):
    """64-bit BLAKE2b of repr(obj): what the store keeps of a reference result (ints, bytes, floats, lists, dicts)"""
    return hashlib.blake2b(repr(obj).encode(), digest_size=8).hexdigest()


class Digest:
    """A reference result known by its digest only (and, for a mapping result, its number of graph chains).
    It equals any value whose digest it is, so `got == want` and diff_results() work on it as on the full value."""

    def __init__(self, h, n_gc=None):
        self.h, self.n_gc = h, n_gc

    def __eq__(self, other):
        return self.h == (other.h if isinstance(other, Digest) else digest(other))

    def __ne__(self, other):
        return not self == other

    __hash__ = None

    def __getitem__(self, k):
        assert k == "n_gc", k
        return self.n_gc

    def __repr__(self):
        return "<reference result %s>" % self.h


_store, _recorded = None, {}


def _record_to(path):
    old = {}
    if os.path.exists(path):
        with open(path) as f:
            old = json.load(f)
    old.update(_recorded)
    with open(path, "w") as f:  # one entry per line
        f.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(old[k], separators=(",", ":"))) for k in sorted(old)) + "\n}\n")


def reference(kind, inputs, compute, stored_form, from_stored):
    """The reference's answer to `inputs`.  With oracle/_ref built: compute() on it (full value, for a detailed diff), checked
    against the stored form when the store has one.  Without: from_stored(the stored form), digests in place of large values.
    MGB_REF_RECORD=<file> adds the stored forms of every computed answer to that JSON file (regenerates the store)."""
    global _store
    if _store is None:
        with open(REF_STORE) as f:
            _store = json.load(f)
    key = digest((kind,) + tuple(inputs))
    if have_ref():
        val = compute()
        rec = json.loads(json.dumps(stored_form(val)))
        assert key not in _store or _store[key] == rec, "%s: the stored reference result differs from the reference's" % kind
        if os.environ.get("MGB_REF_RECORD"):
            if not _recorded:
                atexit.register(_record_to, os.environ["MGB_REF_RECORD"])
            _recorded[key] = rec
        return val
    assert key in _store, "%s: no stored reference result for these inputs (regenerate with oracle/_ref built and MGB_REF_RECORD set)" % kind
    return from_stored(_store[key])


def file_digest(path):
    h = hashlib.blake2b(digest_size=16)
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


def result_form(r):
    """stored form of one mapping result (gchains_to_py), and back"""
    return None if r is None else [digest(r), r["n_gc"]]


def result_from(s):
    return None if s is None else Digest(s[0], s[1])


_ref = None


def load_ref():
    """oracle/_ref/libmgref.so: the unmodified reference compiled as a shared object (test infrastructure)."""
    global _ref
    if _ref is None:
        lib = C.CDLL(REF_SO)
        capi.bind_mapping_api(lib)
        lib.gfa_read.restype = C.POINTER(capi.gfa_t)
        lib.gfa_read.argtypes = [C.c_char_p]
        lib.gfa_destroy.restype = None
        lib.gfa_destroy.argtypes = [C.POINTER(capi.gfa_t)]
        C.c_int.in_dll(lib, "mg_verbose").value = 1
        _ref = lib
    return _ref


_oracle = None


def load_oracle():
    """oracle/liboracle.so: the plain-C restatement of reference functions (oracle/mgoracle.c)"""
    global _oracle
    if _oracle is None:
        subprocess.check_call(["make", "-s", "-C", os.path.join(REPO, "oracle"), "liboracle.so"])
        lib = C.CDLL(os.path.join(REPO, "oracle", "liboracle.so"))
        lib.orc_sketch.restype = C.c_int64
        lib.orc_sketch.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int64]
        lib.orc_radix_sort_128x.restype = None
        lib.orc_radix_sort_128x.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int64]
        lib.orc_hash_str.restype = C.c_uint32
        lib.orc_hash_str.argtypes = [C.c_char_p]
        lib.orc_chain_score.restype = C.c_int32
        lib.orc_chain_score.argtypes = [C.c_uint64] * 4 + [C.c_int32] * 3 + [C.c_float] * 2
        _oracle = lib
    return _oracle


def orc_sketch(orc, seq, w, k, rid):
    cap = len(seq) + 16
    x, y = (C.c_uint64 * cap)(), (C.c_uint64 * cap)()
    n = orc.orc_sketch(seq, len(seq), w, k, rid, x, y, cap)
    assert n <= cap
    return [[x[i], y[i]] for i in range(n)]


_hostsim = None


def load_hostsim():
    global _hostsim
    if _hostsim is None:
        subprocess.check_call(["make", "-s", "-C", os.path.join(REPO, "tests", "hostsim")])
        lib = C.CDLL(HOSTSIM_SO)
        _hostsim = capi.apply_env_params(capi.bind_engine_api(capi.bind_mapping_api(lib)))
    return _hostsim


_hostsim32 = None


def load_hostsim32():
    """the CPU build of the device code with a 32-lane warp simulated by fibres (tests/hostsim/Makefile, mgb_simlanes.h)"""
    global _hostsim32
    if _hostsim32 is None:
        subprocess.check_call(["make", "-s", "-C", os.path.join(REPO, "tests", "hostsim"), "libmgb_hostsim32.so"])
        lib = C.CDLL(os.path.join(REPO, "tests", "hostsim", "libmgb_hostsim32.so"))
        _hostsim32 = capi.apply_env_params(capi.bind_engine_api(capi.bind_mapping_api(lib)))
    return _hostsim32


def read_fasta(fn, upper=True):
    names, seqs = [], []
    cur = []
    with open(fn, "rb") as f:
        for line in f:
            line = line.rstrip(b"\r\n")
            if line.startswith(b">"):
                if names:
                    seqs.append(b"".join(cur))
                names.append(line[1:].split()[0])
                cur = []
            elif names:
                cur.append(line)
    if names:
        seqs.append(b"".join(cur))
    if upper:
        seqs = [s.upper() for s in seqs]
    return names, seqs


def gchains_to_py(p):
    """Everything mg_write_gaf (format.c:121-291) can see, as plain python data."""
    if not p:
        return None
    gs = p.contents
    out = {"n_gc": gs.n_gc, "n_lc": gs.n_lc, "n_a": gs.n_a, "rep_len": gs.rep_len, "gc": [], "lc": [], "a": []}
    for i in range(gs.n_gc):
        g = gs.gc[i]
        d = {k: getattr(g, k) for k in ("id", "parent", "off", "cnt", "n_anchor", "score", "qs", "qe", "plen", "ps", "pe",
                                         "blen", "mlen", "hash", "subsc", "n_sub", "mapq", "flt")}
        d["div"] = C.c_float(g.div).value
        if g.p:
            c = g.p.contents
            d["cigar_hdr"] = (c.n_cigar, c.mlen, c.blen, c.aplen, c.ss, c.ee)
            arr = C.cast(C.addressof(c) + C.sizeof(capi.mg_cigar_t), C.POINTER(C.c_uint64))
            d["cigar"] = [arr[j] for j in range(c.n_cigar)]
        else:
            d["cigar_hdr"], d["cigar"] = None, None
        if g.ds.ds:
            d["ds"] = C.string_at(g.ds.ds, g.ds.len)
            d["ds_off"] = [g.ds.off[j] for j in range(g.ds.n_off)]
        else:
            d["ds"], d["ds_off"] = None, None
        out["gc"].append(d)
    for i in range(gs.n_lc):
        l = gs.lc[i]
        out["lc"].append((l.off, l.cnt, l.v, l.score, l.ed))
    for i in range(gs.n_a):
        out["a"].append((gs.a[i].x, gs.a[i].y))
    return out


def diff_results(a, b):
    """Return a short description of the first difference, or None."""
    if a is None or b is None:
        return None if a is b else "one result is NULL"
    if isinstance(a, Digest) or isinstance(b, Digest):
        return None if a == b else "%r != %r" % (a if isinstance(a, Digest) else digest(a), b if isinstance(b, Digest) else digest(b))
    for k in ("n_gc", "n_lc", "n_a", "rep_len"):
        if a[k] != b[k]:
            return "%s: %r != %r" % (k, a[k], b[k])
    for i, (x, y) in enumerate(zip(a["gc"], b["gc"])):
        for k in x:
            if x[k] != y[k]:
                return "gc[%d].%s: %r != %r" % (i, k, str(x[k])[:200], str(y[k])[:200])
    if a["lc"] != b["lc"]:
        return "lc differs: %r vs %r" % (a["lc"][:8], b["lc"][:8])
    if a["a"] != b["a"]:
        for i, (x, y) in enumerate(zip(a["a"], b["a"])):
            if x != y:
                return "a[%d]: %r != %r" % (i, x, y)
    return None


def map_with_ref(gfa_path, names, seqs, preset="lr", cigar=True, tweak=None):
    """Run the reference's own mg_index/mg_map on every read (CPU).  tweak(mo) may change mapping options after the preset."""
    io, mo = options.opt_set(preset, cigar)
    if tweak:
        tweak(mo)

    def compute():
        ref = load_ref()
        g = ref.gfa_read(gfa_path.encode())
        assert g, "gfa_read failed"
        gi = ref.mg_index(g, C.byref(io), 1, C.byref(mo))
        assert gi
        b = ref.mg_tbuf_init()
        res = []
        for nm, s in zip(names, seqs):
            p = ref.mg_map(gi, len(s), s, b, C.byref(mo), nm)
            res.append(gchains_to_py(p))
            ref.mg_gchain_free(p)
        ref.mg_tbuf_destroy(b)
        ref.mg_idx_destroy(gi)
        ref.gfa_destroy(g)
        return res, mo
    return reference("mg_map", (file_digest(gfa_path), bytes(io), bytes(mo), digest(list(names)), digest(list(seqs))), compute,
                     lambda v: {"mo": bytes(v[1]).hex(), "r": [result_form(r) for r in v[0]]},
                     lambda s: ([result_from(r) for r in s["r"]], capi.mg_mapopt_t.from_buffer_copy(bytes.fromhex(s["mo"]))))


def map_frag_with_ref(gfa_path, frags, preset="lr", cigar=True):
    """The reference's mg_map_frag() on every fragment (name, [segment sequences]): the result of each fragment, which the
    reference returns in its first segment's slot (the others stay NULL)."""
    io, mo = options.opt_set(preset, cigar)

    def compute():
        ref = load_ref()
        ref.mg_map_frag.restype = None
        ref.mg_map_frag.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.POINTER(capi.mg_gchains_t)),
                                    C.c_void_p, C.c_void_p, C.c_char_p]
        g = ref.gfa_read(gfa_path.encode())
        assert g, "gfa_read failed"
        gi = ref.mg_index(g, C.byref(io), 1, C.byref(mo))
        assert gi
        b = ref.mg_tbuf_init()
        res = []
        for nm, parts in frags:
            n_seg = len(parts)
            gcs = (C.POINTER(capi.mg_gchains_t) * n_seg)()
            ref.mg_map_frag(C.cast(gi, C.c_void_p), n_seg, (C.c_int * n_seg)(*[len(x) for x in parts]), (C.c_char_p * n_seg)(*parts), gcs, b,
                            C.cast(C.pointer(mo), C.c_void_p), nm)
            assert all(not gcs[i] for i in range(1, n_seg))
            res.append(gchains_to_py(gcs[0]))
            ref.mg_gchain_free(gcs[0])
        ref.mg_tbuf_destroy(b)
        ref.mg_idx_destroy(gi)
        ref.gfa_destroy(g)
        return res
    return reference("mg_map_frag", (file_digest(gfa_path), bytes(io), bytes(mo), digest(list(frags))), compute,
                     lambda v: [result_form(r) for r in v], lambda s: [result_from(r) for r in s])


def ref_wfa(ts, qs, max_iter, step=None):
    """miniwfa of the reference: mwf_wfa_exact(max_iter); with `step`, mwf_wfa_chain(step) where the exact run gives up
    (score < 0), in the order of mwf_wfa_auto (miniwfa.c:824-834).  Returns (exact run gave up, score, CIGAR)."""
    def compute():
        ref = load_ref()
        mwf_opt_t, mwf_rst_t = _mwf_types()
        opt = mwf_opt_t()
        ref.mwf_opt_init(C.byref(opt))
        opt.flag |= 1
        opt.step, opt.max_iter = 0, max_iter
        rst = mwf_rst_t()
        ref.mwf_wfa_exact(None, C.byref(opt), len(ts), ts, len(qs), qs, C.byref(rst))
        gave_up = rst.s < 0
        if gave_up and step is not None:
            opt.step, opt.max_iter = step, -1
            ref.mwf_wfa_chain(None, C.byref(opt), len(ts), ts, len(qs), qs, C.byref(rst))
        return gave_up, rst.s, [rst.cigar[i] for i in range(rst.n_cigar)]
    return reference("mwf_wfa", (digest(ts), digest(qs), max_iter, step), compute, lambda v: [v[0], v[1], digest(v[2])],
                     lambda s: (s[0], s[1], Digest(s[2])))


_mwf = None


def _mwf_types():
    """ctypes view of miniwfa.h:36-51 (mwf_opt_t, mwf_rst_t) and the prototypes of the reference functions used as the checker"""
    global _mwf
    if _mwf is None:
        ref = load_ref()

        class mwf_opt_t(C.Structure):
            _fields_ = [("flag", C.c_int32), ("x", C.c_int32), ("o1", C.c_int32), ("e1", C.c_int32), ("o2", C.c_int32), ("e2", C.c_int32),
                        ("step", C.c_int32), ("max_s", C.c_int32), ("max_iter", C.c_int64), ("max_occ", C.c_int32), ("kmer", C.c_int32), ("min_len", C.c_int32)]

        class mwf_rst_t(C.Structure):
            _fields_ = [("s", C.c_int32), ("n_cigar", C.c_int32), ("n_iter", C.c_int64), ("cigar", C.POINTER(C.c_uint32))]
        for f in (ref.mwf_wfa_exact, ref.mwf_wfa_chain):
            f.restype = None
            f.argtypes = [C.c_void_p, C.POINTER(mwf_opt_t), C.c_int32, C.c_char_p, C.c_int32, C.c_char_p, C.POINTER(mwf_rst_t)]
        ref.mwf_opt_init.argtypes = [C.POINTER(mwf_opt_t)]
        _mwf = (mwf_opt_t, mwf_rst_t)
    return _mwf


def ref_radix_sort(pairs):
    """klib's radix_sort_128x() of the reference (ksort.h:112-162, not stable) on [(x, y), ...]: the sorted pairs"""
    def compute():
        ref = load_ref()
        ref.radix_sort_128x.restype = None
        ref.radix_sort_128x.argtypes = [C.POINTER(capi.mg128_t), C.POINTER(capi.mg128_t)]
        n = len(pairs)
        a = (capi.mg128_t * n)()
        for i, (x, y) in enumerate(pairs):
            a[i].x, a[i].y = x, y
        ref.radix_sort_128x(a, C.cast(C.byref(a, C.sizeof(a)), C.POINTER(capi.mg128_t)))
        return [(a[i].x, a[i].y) for i in range(n)]
    return reference("radix_sort_128x", (digest(list(pairs)),), compute, digest, Digest)


class mg128_v(C.Structure):
    _fields_ = [("n", C.c_size_t), ("m", C.c_size_t), ("a", C.POINTER(capi.mg128_t))]


def ref_sketch(seq, w, k, rid):
    """mg_sketch() of the reference (sketch.c): the minimizers of `seq` as [[x, y], ...]"""
    def compute():
        ref = load_ref()
        ref.mg_sketch.restype = None
        ref.mg_sketch.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.POINTER(mg128_v)]
        v = mg128_v()
        ref.mg_sketch(None, seq, len(seq), w, k, rid, C.byref(v))
        out = [[v.a[i].x, v.a[i].y] for i in range(v.n)]
        C.CDLL(None).free(v.a)
        return out
    return reference("mg_sketch", (digest(seq), w, k, rid), compute, digest, Digest)


def map_with_engine(lib, gfa_path, names, seqs, preset="lr", cigar=True, gfa_loader=None, tweak=None):
    """Run an engine library (product or hostsim) through mg_index + mg_map_batch."""
    loader = gfa_loader or lib.mgb_gfa_read
    g = loader(gfa_path.encode())
    assert g, "gfa read failed"
    io, mo = options.opt_set(preset, cigar)
    if tweak:
        tweak(mo)
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()
    n = len(seqs)
    qlens = (C.c_int * n)(*[len(s) for s in seqs])
    cseqs = (C.c_char_p * n)(*seqs)
    cnames = (C.c_char_p * n)(*names)
    gcs = (C.POINTER(capi.mg_gchains_t) * n)()
    rc = lib.mg_map_batch(gi, n, qlens, cseqs, cnames, gcs, C.byref(mo))
    assert rc == 0, (rc, lib.mgb_last_error())
    res = []
    for i in range(n):
        res.append(gchains_to_py(gcs[i]))
        lib.mg_gchain_free(gcs[i])
    st = capi.mgb_stats_t()
    lib.mgb_get_stats(gi, C.byref(st))
    lib.mg_idx_destroy(gi)
    return res, mo, st


def gaf_with_engine(lib, gfa_path, names, seqs, preset="lr", cigar=True, flag_extra=0):
    """Map through mg_index + mg_map_batch and format with mgb_write_gaf: the text `minigraph -cx preset` prints."""
    g = lib.mgb_gfa_read(gfa_path.encode())
    assert g, "gfa read failed"
    io, mo = options.opt_set(preset, cigar)
    mo.flag |= flag_extra
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()
    n = len(seqs)
    qlens = (C.c_int * n)(*[len(s) for s in seqs])
    cseqs = (C.c_char_p * n)(*seqs)
    cnames = (C.c_char_p * n)(*names)
    gcs = (C.POINTER(capi.mg_gchains_t) * n)()
    rc = lib.mg_map_batch(gi, n, qlens, cseqs, cnames, gcs, C.byref(mo))
    assert rc == 0, (rc, lib.mgb_last_error())
    buf, ln = C.c_void_p(0), C.c_size_t(0)
    lib.mgb_write_gaf_batch(g, n, gcs, qlens, cnames, mo.flag, 0, C.byref(buf), C.byref(ln), None)
    for i in range(n):
        lib.mg_gchain_free(gcs[i])
    text = C.string_at(buf, ln.value) if buf else b""
    C.CDLL(None).free(buf)
    st = capi.mgb_stats_t()
    lib.mgb_get_stats(gi, C.byref(st))
    lib.mg_idx_destroy(gi)
    lib.mgb_gfa_destroy(g)
    return text, st


def gaf_with_ref_binary(gfa_path, fasta_path, preset="lr", threads=1, extra=()):
    """stdout of the unmodified reference CLI (oracle/_ref/minigraph)."""
    cmd = [REF_BIN, "-cx", preset, "-t", str(threads)] + list(extra) + [gfa_path, fasta_path]
    return subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL).stdout


def write_fasta(fn, names, seqs):
    with open(fn, "wb") as f:
        for n, s in zip(names, seqs):
            f.write(b">" + n + b"\n" + s + b"\n")


def sim_reads(hap_fa, out_fa, n, length, err="ont", seed=11, circular=False):
    cmd = [MGSIM, "reads", "-i", hap_fa, "-n", str(n), "-l", str(length), "-e", err, "-s", str(seed), "-o", out_fa]
    if circular:
        cmd.append("-c")
    subprocess.run(cmd, check=True, stderr=subprocess.DEVNULL)


def sim_graph(prefix, length, n_hap, seed=7):
    subprocess.run([MGSIM, "graph", "-l", str(length), "-n", str(n_hap), "-s", str(seed), "-o", prefix], check=True,
                   stderr=subprocess.DEVNULL)


MT_WALKS = [">MTh0>MTh4001>MTh4502>MTh9505>MTh13014>MTh13516", ">MTh0<MTo3426>MTh4502>MTo8961>MTh9505>MTh13516"]


def sim_mt_haps(out_fa):
    cmd = [MGSIM, "walk", "-g", os.path.join(FIX, "MT.gfa"), "-o", out_fa]
    for w in MT_WALKS:
        cmd += ["-w", w]
    subprocess.run(cmd, check=True)
