#!/usr/bin/env python
"""bench.py -- mapped Gbp/s of the seed-chain-align hot path (BASELINE.json metric) on synthetic long reads.

Default workload = the configuration the targets are quoted on (BASELINE.json configs[2], SURVEY 8d C3): a synthetic MHC-scale
rGFA (5 Mb backbone, 8 haplotypes with SVs) <- 100 000 x 15 kb ONT-error reads, -cx lr -c.  Other workloads: --workload c2
(test/MT.gfa <- 10 000 x 10 kb), c4 (MT-human.fa as a linear graph <- 50 000 x 20 kb HiFi-error reads, -cx asm), c5 (200 Mb rGFA,
3 haplotypes <- 12 kb reads; --reads bounds the sample of the nominal 1 M).

One "step" = one pass of the whole hot path (K1 sketch .. K8 base alignment + ds) over the workload's reads, handed to the library
in mini-batches (<= --mini-batch bases, like the reference's mini_batch_size, gmap.c:174).  With N>1 every rank maps its own read
set (seed + rank) against a replicated index: weak scaling, no data-path collective; the only collective is the all-gather of
per-rank GAF byte counts that fixes output offsets.

  e2e     = bases / wall time through the public C API with HOST buffers: `--pipe` host threads call mg_map_batch() on successive
            mini-batches (pack + H2D, kernels, D2H, mg_gchains_t assembly inside every call) and one more thread turns the
            results into GAF text in input order (mgb_write_gaf_batch) -- the reference's kt_pipeline (gmap.c:176-177) in shape
  value   = bases / device time of the kernels alone (CUDA events inside libmgb200, first kernel start to last kernel end of each
            mini-batch, mini-batches run one after the other, reads resident in HBM), measured in a second pass over the same K steps
  roofline= chaining kernel (K4/K5, `k_chain`): algorithmic bytes (16 B/seed in + 16 B/anchor out + 8 B/chain) / its event time
            against MEASURED_PEAKS.json hbm_gbs
  --impl reference : the unmodified reference CLI (oracle/_ref/minigraph -t <all cores>) on the same reads
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import queue
import re
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

FIX = os.path.join(REPO, "tests", "golden", "fixtures")
MGSIM = os.path.join(REPO, "tools", "mgsim")
REF_BIN = os.path.join(REPO, "oracle", "_ref", "minigraph")
MT_WALKS = [">MTh0>MTh4001>MTh4502>MTh9505>MTh13014>MTh13516", ">MTh0<MTo3426>MTh4502>MTo8961>MTh9505>MTh13516"]

# name -> (default reads, read length, preset, error model, description of graph)
WORKLOADS = {
    "c2": (10000, 10000, "lr", "ont", "test/MT.gfa"),
    "c3": (100000, 15000, "lr", "ont", "synthetic MHC-scale rGFA (5 Mb backbone, 8 haplotypes with SVs, mgsim seed 7)"),
    "c4": (50000, 20000, "asm", "hifi", "test/MT-human.fa as a linear graph (reads from the circularised sequence)"),
    "c5": (100000, 12000, "lr", "ont", "synthetic 200 Mb rGFA (3 haplotypes with SVs, mgsim seed 17)"),
}
REF_BUDGET_S = 240.0  # the reference arm sizes its per-step sample so that W + K steps end within about this


def sh(cmd, **kw):
    subprocess.run(cmd, check=True, stderr=subprocess.DEVNULL, **kw)


def make_workload(name, tmp, rank, n_reads):
    """Deterministic inputs (mgsim: splitmix64 seeded as SURVEY 8d states).  Returns (graph path, reads FASTA path)."""
    _, rlen, _, err, _ = WORKLOADS[name]
    reads = os.path.join(tmp, "%s.reads.%d.fa" % (name, rank))
    if name == "c2":
        hap = os.path.join(tmp, "mt.hap.fa")
        cmd = [MGSIM, "walk", "-g", os.path.join(FIX, "MT.gfa"), "-o", hap]
        for w in MT_WALKS:
            cmd += ["-w", w]
        sh(cmd)
        sh([MGSIM, "reads", "-i", hap, "-n", str(n_reads), "-l", str(rlen), "-e", err, "-s", str(11 + rank), "-o", reads])
        return os.path.join(FIX, "MT.gfa"), reads
    if name == "c4":
        gfa = os.path.join(FIX, "MT-human.fa")
        sh([MGSIM, "reads", "-i", gfa, "-n", str(n_reads), "-l", str(rlen), "-e", err, "-s", str(13 + rank), "-o", reads, "-c"])
        return gfa, reads
    glen, nhap, gseed, rseed = (5000000, 8, 7, 5) if name == "c3" else (200000000, 3, 17, 19)
    prefix = os.path.join(tmp, name)
    if not os.path.exists(prefix + ".gfa"):
        sh([MGSIM, "graph", "-l", str(glen), "-n", str(nhap), "-s", str(gseed), "-o", prefix])
    sh([MGSIM, "reads", "-i", prefix + ".hap.fa", "-n", str(n_reads), "-l", str(rlen), "-e", err, "-s", str(rseed + rank), "-o", reads])
    return prefix + ".gfa", reads


def workload_text(name, n_reads):
    _, rlen, preset, err, graph = WORKLOADS[name]
    errs = "ONT-error (4% sub, 3% del, 3% ins)" if err == "ont" else "HiFi-error (0.2% sub, 0.15% del, 0.15% ins)"
    note = "; a bounded sample of the configuration's 1 000 000 reads" if name == "c5" and n_reads < 1000000 else ""
    return "%s <- %d x %d bp synthetic %s reads (mgsim, seed + rank)%s, -cx %s -c" % (graph, n_reads, rlen, errs, note, preset)


def read_fasta(fn):
    with open(fn, "rb") as f:
        data = f.read().split(b"\n")
    return [data[i][1:] for i in range(0, len(data) - 1, 2)], [data[i + 1] for i in range(0, len(data) - 1, 2)]


def write_fasta(fn, names, seqs):
    with open(fn, "wb") as f:
        f.write(b"".join(b">" + n + b"\n" + s + b"\n" for n, s in zip(names, seqs)))


def run_reference_cli(gfa, fasta, preset, threads, out=None):
    """Mapping-phase seconds of the reference (BASELINE.md section 3: last 'mapped' stamp minus the 'indexed' stamp)."""
    t0 = time.perf_counter()
    with open(out, "wb") if out else open(os.devnull, "wb") as fo:
        p = subprocess.run([REF_BIN, "-cx", preset, "-t", str(threads), gfa, fasta], stdout=fo, stderr=subprocess.PIPE, check=True)
    wall = time.perf_counter() - t0
    log = p.stderr.decode()
    t_idx = re.findall(r"\[M::mg_index::([0-9.]+)\*", log)
    t_map = re.findall(r"\[M::worker_pipeline::([0-9.]+)\*[0-9.]+\] mapped", log)
    if t_idx and t_map:
        return float(t_map[-1]) - float(t_idx[-1]), wall
    return wall, wall


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=5).stdout.decode().strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(self.rows)}


def chain_traffic(workload):
    """DRAM bytes of the chaining kernels (k_chain + k_chain_rescue, one launch each = one mini-batch) from the newest committed
    `ncu --set full` digests of this workload (profiles/r*<workload>_ncu_k_chain*.txt), or (None, None)."""
    import glob
    tot, srcs = 0.0, []
    for kern in ("k_chain", "k_chain_rescue"):
        fns = sorted(glob.glob(os.path.join(REPO, "profiles", "r*%s_ncu_%s.txt" % (workload, kern))), reverse=True)
        if not fns:
            return None, None
        rd = wr = None
        with open(fns[0]) as f:
            for ln in f:
                t = ln.rstrip("\n").split("\t")
                if len(t) == 3 and t[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    v = float(t[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[t[2]]
                    if t[0].startswith("dram__bytes_read"):
                        rd = v
                    else:
                        wr = v
        if rd is None or wr is None:
            return None, None
        tot += rd + wr
        srcs.append(os.path.relpath(fns[0], REPO))
    return tot, " + ".join(srcs)


def hbm_peak():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def mini_batches(lens, max_bases):
    """Contiguous [lo, hi) ranges of at most max_bases bases, of similar size."""
    tot = sum(lens)
    m = max(1, -(-tot // max_bases))
    out, lo, acc, k = [], 0, 0, 1
    for i, l in enumerate(lens):
        acc += l
        if k < m and acc >= tot * k / m:
            out.append((lo, i + 1))
            lo, k = i + 1, k + 1
    if lo < len(lens):
        out.append((lo, len(lens)))
    return out


DUMP_BUDGET = 64000000  # bytes of all --dump-outputs arrays together


def dump_outputs(out_dir, n, result_of):
    """Write what mg_map_batch() returned for a fixed, seeded sample of the n reads as out_dir/<name>.npy.  Reads are taken in
    the order of a seeded permutation while all arrays together stay within DUMP_BUDGET bytes; rows are in read order and
    "row" columns number the reads (or graph chains) of the sample from 0.  float64 holds every integer exactly: 64-bit
    anchors are split into 32-bit halves.  result_of(i) is the mg_gchains_t pointer of read i (NULL: no result object).
      read_index [R]      read number in the input
      reads      [R, 4]   n_gc, n_lc, n_a, rep_len (all -1: no result object)
      gchains    [G, 28]  read row, id, parent, off, cnt, n_anchor, score, qs, qe, plen, ps, pe, blen, mlen, div, hash, subsc, n_sub,
                          mapq, flt, n_cigar, cigar mlen, blen, aplen, ss, ee (-1 from n_cigar on: no CIGAR), ds len, n_off (-1: no ds)
      cigar      [C, 3]   gchain row, operation length, operation code
      lchains    [L, 6]   read row, off, cnt, v, score, ed
      anchors    [A, 5]   read row, x >> 32, x & 0xffffffff, y >> 32, y & 0xffffffff
      ds         [D]      the ds strings of the graph chains in gchain order, one byte per element (float32)
      ds_off     [O, 2]   gchain row, offset
    Returns (number of reads written, bytes written)."""
    import random
    import numpy as np
    from minigraph_b200 import capi

    def size_of(p):  # bytes the read adds to the arrays
        if not p:
            return 8 * 5
        gs, b = p.contents, 8 * (5 + 6 * p.contents.n_lc + 5 * p.contents.n_a)
        for j in range(gs.n_gc):
            g = gs.gc[j]
            b += 8 * 28 + (24 * g.p.contents.n_cigar if g.p else 0) + (4 * g.ds.len + 16 * g.ds.n_off if g.ds.ds else 0)
        return b
    picked, total = [], 8 * 128  # the .npy headers
    for i in random.Random(12345).sample(range(n), n):
        b = size_of(result_of(i))
        if total + b > DUMP_BUDGET:
            break
        picked.append(i)
        total += b
    picked.sort()
    out = {k: [] for k in ("reads", "gchains", "cigar", "lchains", "anchors", "ds", "ds_off")}
    n_gc_rows = 0
    for r, i in enumerate(picked):
        p = result_of(i)
        if not p:
            out["reads"].append(np.full((1, 4), -1.0))
            continue
        gs = p.contents
        out["reads"].append(np.array([[gs.n_gc, gs.n_lc, gs.n_a, gs.rep_len]], dtype=np.float64))
        for j in range(gs.n_gc):
            g, row = gs.gc[j], n_gc_rows + j
            cols = [r, g.id, g.parent, g.off, g.cnt, g.n_anchor, g.score, g.qs, g.qe, g.plen, g.ps, g.pe, g.blen, g.mlen, g.div, g.hash,
                    g.subsc, g.n_sub, g.mapq, g.flt]
            if g.p:
                c = g.p.contents
                cols += [c.n_cigar, c.mlen, c.blen, c.aplen, c.ss, c.ee]
                ops = np.frombuffer((C.c_uint64 * c.n_cigar).from_address(C.addressof(c) + C.sizeof(capi.mg_cigar_t)), dtype=np.uint64)
                out["cigar"].append(np.stack([np.full(c.n_cigar, float(row)), (ops >> np.uint64(4)).astype(np.float64),
                                              (ops & np.uint64(15)).astype(np.float64)], axis=1))
            else:
                cols += [-1] * 6
            if g.ds.ds:
                cols += [g.ds.len, g.ds.n_off]
                out["ds"].append(np.frombuffer(C.string_at(g.ds.ds, g.ds.len), dtype=np.uint8).astype(np.float32))
                offs = np.ctypeslib.as_array(g.ds.off, shape=(g.ds.n_off,)).astype(np.float64) if g.ds.n_off else np.zeros(0)
                out["ds_off"].append(np.stack([np.full(g.ds.n_off, float(row)), offs], axis=1))
            else:
                cols += [-1, -1]
            out["gchains"].append(np.array([cols], dtype=np.float64))
        n_gc_rows += gs.n_gc
        for j in range(gs.n_lc):
            lc = gs.lc[j]
            out["lchains"].append(np.array([[r, lc.off, lc.cnt, lc.v, lc.score, lc.ed]], dtype=np.float64))
        if gs.n_a > 0:
            a = np.frombuffer((C.c_uint64 * (2 * gs.n_a)).from_address(C.addressof(gs.a.contents)), dtype=np.uint64).reshape(-1, 2)
            hi, lo = (a >> np.uint64(32)).astype(np.float64), (a & np.uint64(0xffffffff)).astype(np.float64)
            out["anchors"].append(np.stack([np.full(gs.n_a, float(r)), hi[:, 0], lo[:, 0], hi[:, 1], lo[:, 1]], axis=1))
    width = {"reads": 4, "gchains": 28, "cigar": 3, "lchains": 6, "anchors": 5, "ds_off": 2}
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"read_index": np.array(picked, dtype=np.float64)}
    for k, v in out.items():
        empty = np.zeros(0, dtype=np.float32) if k == "ds" else np.zeros((0, width[k]))
        arrays[k] = np.concatenate(v) if v else empty
    written = 0
    for k, v in arrays.items():
        fn = os.path.join(out_dir, k + ".npy")
        np.save(fn, v)
        written += os.path.getsize(fn)
    assert written <= DUMP_BUDGET, written
    return len(picked), written


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mgb200")
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU (default: the workload's own number)")
    ap.add_argument("--mini-batch", type=int, default=400000000, help="bases per mg_map_batch() call")
    ap.add_argument("--pipe", type=int, default=3, help="host threads calling mg_map_batch() at once")
    ap.add_argument("--no-cpu", action="store_true", help="skip the reference run on the host cores (no cpu_baseline, no parity check): profiling runs")
    ap.add_argument("--check", default="all", help="'all': after the timed region the GAF text of every read of rank 0 is compared with the reference binary's, byte for byte; N: the first N reads; 0: skip")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned for a seeded sample of rank 0's reads "
                    "as DIR/<name>.npy (float32/float64, at most 64 MB; see dump_outputs) to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    # stdout carries exactly one JSON line: everything libraries print to fd 1 (NCCL's version banner, ...) goes to stderr instead
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    tmp = tempfile.mkdtemp(prefix="mgb_bench_")
    ncores = os.cpu_count() or 1
    n_reads = a.reads or WORKLOADS[a.workload][0]
    preset = WORKLOADS[a.workload][2]
    metric = "mapped Gbp/s (-cx %s)" % preset

    def config_of(n, bases):  # identical in both arms
        return {"workload": workload_text(a.workload, n_reads), "reads_per_gpu": n, "bases_per_gpu": bases,
                "l2": "inputs (%.0f MB of reads per step) are larger than L2; no flush needed" % (bases / 1e6) if bases > 400e6 else "512 MiB flush buffer written between steps"}

    if a.impl == "reference":
        if rank != 0:
            return
        gfa, fa = make_workload(a.workload, tmp, 0, n_reads)
        names, seqs = read_fasta(fa)
        n, bases = len(seqs), sum(len(s) for s in seqs)
        # size the per-step sample: a first run on 4 % of the reads gives the rate of this box
        probe = max(200, n // 25)
        pfa = os.path.join(tmp, "probe.fa")
        write_fasta(pfa, names[:probe], seqs[:probe])
        run_reference_cli(gfa, pfa, preset, ncores)
        t_probe = run_reference_cli(gfa, pfa, preset, ncores)[0]
        rate = sum(len(s) for s in seqs[:probe]) / max(t_probe, 1e-3)
        runs = a.steps + a.warmup
        per_step = int(min(n, max(n // 8, (rate * REF_BUDGET_S / max(runs, 1)) / (bases / n))))
        if per_step >= n * 0.9:
            per_step = n
        # step i maps reads [i*per_step, (i+1)*per_step) modulo n: the steps rotate through the SAME input the GPU arm maps
        def sample_file(i):
            if per_step == n:
                return fa, bases
            lo = (i * per_step) % n
            idx = [(lo + j) % n for j in range(per_step)]
            fn = os.path.join(tmp, "step.fa")
            write_fasta(fn, [names[j] for j in idx], [seqs[j] for j in idx])
            return fn, sum(len(seqs[j]) for j in idx)
        for i in range(a.warmup):
            fn, _ = sample_file(i)
            run_reference_cli(gfa, fn, preset, ncores)
        ts, bs = [], []
        for i in range(a.steps):
            fn, b = sample_file(a.warmup + i)
            ts.append(run_reference_cli(gfa, fn, preset, ncores)[0])
            bs.append(b)
        v = sum(bs) / sum(ts) / 1e9
        rates = sorted(b / t / 1e9 for b, t in zip(bs, ts))
        sample = ("all %d reads (%.0f Mbp) every step" % (n, bases / 1e6)) if per_step == n else \
            "%d of the %d reads (%.0f Mbp) per step, rotating through the input (%d steps cover it %.1f times); sized from a probe run so that %d runs end in about %d s" % (
                per_step, n, sum(bs) / len(bs) / 1e6, a.steps, a.steps * per_step / n, runs, REF_BUDGET_S)
        sample += "; mapping phase (index-ready to last 'mapped' stamp) of `oracle/_ref/minigraph -cx %s -t %d`, page cache warm" % (preset, ncores)
        json_out.write(json.dumps({
            "impl": "reference", "metric": metric, "value": v, "unit": "Gbp/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": sum(ts) / len(ts) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/u8 (fp32 chain penalties)",
            "data": "synthetic", "config": config_of(n, bases), "same_reads_as_gpu_arm": True, "reads_per_step": per_step,
            "value_median_of_steps": rates[len(rates) // 2], "value_min_max": [rates[0], rates[-1]], "host_cores": ncores,
            "cpu_baseline": {"value": v, "unit": "Gbp/s", "cores": ncores, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }) + "\n")
        json_out.flush()
        return

    import torch
    import torch.distributed as dist
    from minigraph_b200 import capi, options
    dry = bool(os.environ.get("MGB_BENCH_DRY"))  # development only: the control flow of this script against the CPU simulator of the tests (no GPU, no valid numbers)
    if dry:
        import mgtest
        torch.cuda.synchronize = lambda: None
    else:
        torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = mgtest.load_hostsim() if dry else capi.load_product()  # applies MGB_PARAMS (engine switches for experiments)
    lib.mgb_set_param(b"device", local_rank)
    n_pipe = max(1, a.pipe)
    lib.mgb_set_param(b"slots", n_pipe)
    # this rank's share of the host cores: n_pipe mapping threads (packing, result assembly) and the GAF writer run at once
    share = max(4, ncores // world)
    host_threads = max(2, min(32, share // (n_pipe + 1)))
    gaf_threads = max(2, min(48, share - n_pipe * host_threads // 2))
    lib.mgb_set_param(b"host_threads", host_threads)
    gfa, fa = make_workload(a.workload, tmp, rank, n_reads)
    rd = lib.mgb_reads_load(fa.encode(), 0)  # the library's own FASTA reader (input side of the path; not in the timed region)
    assert rd, fa
    n = int(rd.contents.n_reads)
    qlens, cseqs, cnames = rd.contents.len, rd.contents.seq, rd.contents.name
    lens = qlens[:n]
    bases = int(rd.contents.n_bases)
    g = lib.mgb_gfa_read(gfa.encode())
    io, mo = options.opt_set(preset, cigar=True)
    t0 = time.perf_counter()
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()
    t_index = time.perf_counter() - t0
    mbs = mini_batches(lens, a.mini_batch)
    M = len(mbs)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda") if bases <= 400e6 and not dry else None

    def sub(arr, ctype, lo):
        return C.cast(C.addressof(arr.contents) + lo * C.sizeof(ctype), C.POINTER(ctype))

    # GAF text buffers, one per mini-batch of a step (reused every step): after the run they hold the text of the last step
    gaf_buf = [C.c_void_p(0) for _ in range(M)]
    gaf_cap = [C.c_size_t(0) for _ in range(M)]
    gaf_len = [C.c_size_t(0) for _ in range(M)]
    acc = {"pack": 0.0, "h2d": 0.0, "d2h": 0.0, "asm": 0.0, "call": 0.0, "gaf": 0.0, "span": 0.0, "chain": 0.0, "launches": 0, "retry": 0,
           "w_slot": 0.0, "w_gpu": 0.0, "w_up": 0.0, "w_pass": 0.0, "w_redo": 0.0, "w_down": 0.0,
           "seeds": 0, "anchors": 0, "chains": 0, "out_bytes": 0, "lab_new": 0, "jobs": 0}
    acc_lock = threading.Lock()
    kern = [0.0] * 10
    last_st = capi.mgb_stats_t()

    last = {}  # --dump-outputs: mini-batch -> results of the last step of the last timed region, freed once written out

    def run_steps(n_steps, pipelined, record, keep_last=False):
        """n_steps passes over the reads.  pipelined: n_pipe threads map successive mini-batches, a writer formats them in order.
        keep_last: the writer keeps the results of the last step in `last` instead of freeing them."""
        jobs = [(s, k) for s in range(n_steps) for k in range(M)]
        results = queue.Queue(maxsize=2 * n_pipe + 2)
        nxt = [0]
        nxt_lock = threading.Lock()
        errs = []

        def mapper():
            st = capi.mgb_stats_t()
            while True:
                with nxt_lock:
                    j = nxt[0]
                    nxt[0] += 1
                if j >= len(jobs) or errs:
                    return
                lo, hi = mbs[jobs[j][1]]
                gcs = (C.POINTER(capi.mg_gchains_t) * (hi - lo))()
                if flush is not None:
                    flush.fill_(1)
                t0 = time.perf_counter()
                rc = lib.mg_map_batch(gi, hi - lo, sub(qlens, C.c_int, lo), sub(cseqs, C.c_char_p, lo), sub(cnames, C.c_char_p, lo), gcs, C.byref(mo))
                dt = (time.perf_counter() - t0) * 1e3
                if rc != 0:
                    errs.append(lib.mgb_last_error())
                    results.put((j, None))
                    return
                lib.mgb_get_stats(gi, C.byref(st))
                if record:
                    with acc_lock:
                        acc["pack"] += st.t_pack_ms; acc["h2d"] += st.t_h2d_ms; acc["d2h"] += st.t_d2h_ms; acc["asm"] += st.t_asm_ms; acc["call"] += dt
                        acc["span"] += st.t_dev_span_ms; acc["chain"] += st.t_kernel_ms[1]; acc["launches"] += st.n_launches
                        acc["seeds"] += st.n_seeds; acc["anchors"] += st.n_anchors_out; acc["chains"] += st.n_chains_out
                        acc["out_bytes"] += st.out_bytes; acc["lab_new"] += st.n_lab_new; acc["jobs"] += st.n_jobs; acc["retry"] += st.n_retry
                        acc["w_slot"] += st.w_slot_wait_ms; acc["w_gpu"] += st.w_gpu_wait_ms; acc["w_up"] += st.w_upload_ms; acc["w_pass"] += st.w_pass_ms; acc["w_redo"] += st.w_redo_ms; acc["w_down"] += st.w_download_ms
                        for i in range(10):
                            kern[i] += st.t_kernel_ms[i]
                        C.memmove(C.byref(last_st), C.byref(st), C.sizeof(st))
                results.put((j, gcs))

        def writer():
            pending, want = {}, 0
            while want < len(jobs):
                j, gcs = results.get()
                if gcs is None:
                    return
                pending[j] = gcs
                while want in pending:
                    gcs = pending.pop(want)
                    k = jobs[want][1]
                    lo, hi = mbs[k]
                    t0 = time.perf_counter()
                    lib.mgb_write_gaf_batch(g, hi - lo, gcs, sub(qlens, C.c_int, lo), sub(cnames, C.c_char_p, lo), mo.flag, gaf_threads,
                                            C.byref(gaf_buf[k]), C.byref(gaf_len[k]), C.byref(gaf_cap[k]))
                    if keep_last and jobs[want][0] == n_steps - 1:
                        last[k] = gcs
                    else:
                        lib.mgb_free_batch(hi - lo, gcs)
                    if record:
                        acc["gaf"] += (time.perf_counter() - t0) * 1e3
                    want += 1

        th = [threading.Thread(target=mapper) for _ in range(n_pipe if pipelined else 1)] + [threading.Thread(target=writer)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert not errs, errs

    run_steps(a.warmup, True, False)
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- timed region 1: end to end through the public API, pipelined ----
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_begin = time.perf_counter()
    run_steps(a.steps, True, True)
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_begin
    if world > 1:
        dist.barrier()
    e2e_acc = dict(acc)
    kern_e2e = list(kern)
    # ---- timed region 2: the kernels alone (CUDA events), mini-batches one after the other ----
    for k in acc:
        acc[k] = 0
    kern[:] = [0.0] * 10
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    run_steps(a.steps, False, True, keep_last=bool(a.dump_outputs) and rank == 0)
    torch.cuda.synchronize()
    t_kern = acc["span"] / 1e3
    if world > 1:
        dist.barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    gaf_bytes = sum(x.value for x in gaf_len)
    # the one collective of the path: per-rank GAF byte counts -> output offsets (SURVEY section 8e)
    from minigraph_b200 import dist as mdist
    my_off, counts = mdist.gaf_offsets(gaf_bytes, device=None if dry else "cuda")
    offsets = [sum(counts[:i]) for i in range(len(counts))]
    if world > 1:
        tm = torch.tensor([t_kern, t_wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        t_kern, t_wall = float(tm[0].item()), float(tm[1].item())
    total_bases = bases * world
    value = total_bases * a.steps / t_kern / 1e9
    e2e = total_bases * a.steps / t_wall / 1e9
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    dumped = None
    if a.dump_outputs:
        def result_of(i):
            k = next(k for k, (lo, hi) in enumerate(mbs) if lo <= i < hi)
            return last[k][i - mbs[k][0]]
        n_dump, dump_bytes = dump_outputs(a.dump_outputs, n, result_of)
        for k, (lo, hi) in enumerate(mbs):
            lib.mgb_free_batch(hi - lo, last[k])
        dumped = {"dir": a.dump_outputs, "reads": n_dump, "bytes": dump_bytes}

    # ---- untimed: the reference on the host cores, once: CPU baseline and, from its output, the parity check ----
    check, cpu = None, None
    n_chk = 0 if a.no_cpu or a.check == "0" else (n if a.check == "all" else min(n, int(a.check)))
    if n_chk > 0 and os.path.exists(REF_BIN):
        try:
            cfa = fa
            if n_chk < n:
                cfa = os.path.join(tmp, "check.fa")
                write_fasta(cfa, [cnames[i] for i in range(n_chk)], [C.string_at(cseqs[i], lens[i]) for i in range(n_chk)])
            pfa = os.path.join(tmp, "warm.fa")
            write_fasta(pfa, [cnames[i] for i in range(min(n, 200))], [C.string_at(cseqs[i], lens[i]) for i in range(min(n, 200))])
            run_reference_cli(gfa, pfa, preset, ncores)  # binary and graph into the page cache
            out_fn = os.path.join(tmp, "ref.gaf")
            tcpu, _ = run_reference_cli(gfa, cfa, preset, ncores, out=out_fn)
            cb = sum(lens[:n_chk])
            cpu = {"value": cb / tcpu / 1e9, "unit": "Gbp/s", "cores": ncores, "kind": "reference",
                   "sample": "%s %d reads of rank 0 (%.0f Mbp), one run, mapping phase of `oracle/_ref/minigraph -cx %s -t %d`; `--impl reference` repeats it K times" % (
                       "all" if n_chk == n else "the first", n_chk, cb / 1e6, preset, ncores)}
            with open(out_fn, "rb") as f:
                want = f.read()
            got = b"".join(C.string_at(gaf_buf[k], gaf_len[k].value) for k in range(M))
            if n_chk < n:  # the text of the first n_chk reads: lines are in read order, a read may have several or (unmapped) one
                m = re.search(rb"^" + re.escape(cnames[n_chk]) + rb"\t", got, re.M)
                got = got[:m.start()] if m else got
            check = {"reads": n_chk, "gaf_bytes": len(want), "identical": got == want, "md5": hashlib.md5(got).hexdigest()}
        except Exception as e:  # the measured line is still worth printing; the failure is reported in it
            check = {"reads": 0, "identical": False, "error": repr(e)[:200]}

    peak, peak_src = hbm_peak()
    chain_bytes = 16.0 * acc["seeds"] + 16.0 * acc["anchors"] + 8.0 * acc["chains"]  # over all launches of the second region
    n_launch_chain = a.steps * M
    t_chain = acc["chain"] / 1e3
    achieved = chain_bytes / t_chain / 1e9 if t_chain > 0 else 0.0
    traffic, traffic_src = chain_traffic(a.workload)
    st = last_st
    out = {
        "metric": metric, "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": t_kern / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64/u8 (fp32 chain penalties, bit-exact)", "data": "synthetic",
        "config": config_of(n, bases),
        "parallelism": "reads sharded one read set per GPU, index replicated; all-gather of GAF byte counts only", "gaf_offsets": offsets,
        "mini_batches_per_step": M, "pipe_threads": n_pipe, "host_threads": host_threads, "gaf_threads": gaf_threads, "host_cores": ncores,
        "engine_params": capi.env_params(), "index_build_s": t_index,
        "kernel_ms_per_step": {k: round(kern[i] / a.steps, 3) for i, k in enumerate(capi.KERNEL_NAMES) if k != "k_index_sketch"},
        "kernel_ms_per_step_in_e2e_region": {k: round(kern_e2e[i] / a.steps, 3) for i, k in enumerate(capi.KERNEL_NAMES) if k != "k_index_sketch"},
        "kernel_ms_note": "CUDA-event time of each kernel summed over the %d mini-batches of a step, second timed region (kernels of one mini-batch at a time)" % M,
        "wfa_jobs_per_step": acc["jobs"] // a.steps, "label_sources_new_in_timed_steps": acc["lab_new"],
        "e2e": {"value": e2e, "unit": "Gbp/s", "ms_per_step": t_wall / a.steps * 1e3,
                "h2d_bytes_per_step": int(bases + 32 * n), "d2h_bytes_per_step": int(e2e_acc["out_bytes"] // a.steps + 144 * n),
                "includes": "wall clock of K steps: %d host threads call mg_map_batch() on successive mini-batches (host buffers in: pack + H2D, all kernels, D2H of result blobs, mg_gchains_t assembly) "
                            "while one thread writes the GAF text (%d bytes/step) of finished mini-batches in input order and frees the results" % (n_pipe, gaf_bytes)},
        "host_ms_per_step": {"pack": e2e_acc["pack"] / a.steps, "h2d": e2e_acc["h2d"] / a.steps, "d2h": e2e_acc["d2h"] / a.steps, "assemble": e2e_acc["asm"] / a.steps,
                             "mg_map_batch_calls(sum over threads)": e2e_acc["call"] / a.steps, "gaf_text(writer thread)": e2e_acc["gaf"] / a.steps,
                             "call_wall_parts(sum over threads)": {"wait_for_slot": e2e_acc["w_slot"] / a.steps, "pack+h2d": e2e_acc["w_up"] / a.steps, "wait_for_gpu": e2e_acc["w_gpu"] / a.steps, "kernels+syncs": e2e_acc["w_pass"] / a.steps,
                                                                   "large_arena_redo": e2e_acc["w_redo"] / a.steps, "pack_results+d2h": e2e_acc["w_down"] / a.steps, "device_span": e2e_acc["span"] / a.steps},
                             "reads_redone_with_large_arena": e2e_acc["retry"] / a.steps},
        "device_cycles_last_call": {k: (int(st.prof[i]) >> 16 if k in ("wfa_max_cyc", "gwfa_max_cyc") else int(st.prof[i])) for i, k in enumerate(capi.PROF_NAMES)},
        "arena_peak_bytes_last_call": int(st.arena_peak),
        "wfa_tier_routing": {"skip_tier1_at": int(st.skip1_len), "skip_tier2_at": int(st.skip2_len)},
        "gpu_launches": int(e2e_acc["launches"]),
        "roofline": {"kernel": "k_chain (linear chaining: mg_lchain_dp/rmq + backtrack + compaction)", "bound": "hbm", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": chain_bytes / n_launch_chain, "launch_ms": t_chain / n_launch_chain * 1e3, "launches_timed": n_launch_chain,
                     "peak_source": peak_src,
                     "bytes_model": "16 B x %d seeds in + 16 B x %d anchors out + 8 B x %d chains over %d launches" % (acc["seeds"], acc["anchors"], acc["chains"], n_launch_chain)},
        "cpu_baseline": cpu, "parity_check": check,
        "clocks": sampler.summary(),
    }
    if dumped:
        out["outputs_dumped"] = dumped
    if dry:
        out["INVALID"] = "MGB_BENCH_DRY: CPU simulator, not a measurement"
    json_out.write(json.dumps(out) + "\n")
    json_out.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
