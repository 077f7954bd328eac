"""Two routes from reads to GAF text, measured in one process, step by step in turn, on bench.py's workload.

  A  objects:  --pipe threads call mg_map_batch(); one writer thread calls mgb_write_gaf_batch() + mgb_free_batch() in input order
               (bench.py's end-to-end region)
  B  text:     --pipe threads call mgb_map_batch_gaf(), which formats the text on the device

Every step's text (its mini-batches in input order) must have the same md5 in both routes, or the run fails.  Prints one JSON line
per route, with the GPU's name, power limit and maximum SM clock as nvidia-smi reports them in the same run.

    python tools/gaf_route_bench.py --workload c3 --steps 3 --warmup 1 [--out FILE]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import resource
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench  # noqa: E402
from minigraph_b200 import capi, options  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def cpu_s():
    u = resource.getrusage(resource.RUSAGE_SELF)
    return u.ru_utime + u.ru_stime


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--reads", type=int, default=0, help="reads (default: the workload's own number)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--pipe", type=int, default=3, help="host threads mapping at once")
    ap.add_argument("--mini-batch", type=int, default=400000000, help="bases per call")
    ap.add_argument("--out", help="also write the JSON lines to this file")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    lib = capi.load_product()
    n_pipe = max(1, a.pipe)
    ncores = os.cpu_count() or 1
    host_threads = max(2, min(32, max(4, ncores) // (n_pipe + 1)))  # bench.py's split of the host cores
    gaf_threads = max(2, min(48, max(4, ncores) - n_pipe * host_threads // 2))
    lib.mgb_set_param(b"slots", n_pipe)
    lib.mgb_set_param(b"host_threads", host_threads)
    tmp = tempfile.mkdtemp(prefix="mgb_gafroute_")
    n_reads = a.reads or bench.WORKLOADS[a.workload][0]
    preset = bench.WORKLOADS[a.workload][2]
    gfa, fa = bench.make_workload(a.workload, tmp, 0, n_reads)
    rd = lib.mgb_reads_load(fa.encode(), 0)
    assert rd, fa
    n, bases = int(rd.contents.n_reads), int(rd.contents.n_bases)
    qlens, cseqs, cnames = rd.contents.len, rd.contents.seq, rd.contents.name
    mbs = bench.mini_batches(qlens[:n], a.mini_batch)
    M = len(mbs)
    g = lib.mgb_gfa_read(gfa.encode())
    io, mo = options.opt_set(preset, cigar=True)
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi, lib.mgb_last_error()

    def sub(arr, ctype, lo):
        return C.cast(C.addressof(arr.contents) + lo * C.sizeof(ctype), C.POINTER(ctype))

    bufs = {r: ([C.c_void_p(0) for _ in range(M)], [C.c_size_t(0) for _ in range(M)], [C.c_size_t(0) for _ in range(M)]) for r in "AB"}

    def step(route):
        """one pass over the reads; returns (wall ms, host CPU s, md5 of the text, sums of the per-call stats, writer ms)"""
        buf, ln, cap = bufs[route]
        nxt, lock, errs = [0], threading.Lock(), []
        tot = {"out_bytes": 0, "t_dev_span_ms": 0.0, "t_gaf_ms": 0.0, "t_asm_ms": 0.0, "n_launches": 0}
        done = {}
        cv = threading.Condition()
        writer_ms = [0.0]

        def mapper():
            st = capi.mgb_stats_t()
            while True:
                with lock:
                    k = nxt[0]
                    nxt[0] += 1
                if k >= M or errs:
                    return
                lo, hi = mbs[k]
                if route == "A":
                    gcs = (C.POINTER(capi.mg_gchains_t) * (hi - lo))()
                    rc = lib.mg_map_batch(gi, hi - lo, sub(qlens, C.c_int, lo), sub(cseqs, C.c_char_p, lo), sub(cnames, C.c_char_p, lo), gcs, C.byref(mo))
                else:
                    gcs = None
                    rc = lib.mgb_map_batch_gaf(gi, hi - lo, sub(qlens, C.c_int, lo), sub(cseqs, C.c_char_p, lo), sub(cnames, C.c_char_p, lo), C.byref(mo),
                                               C.byref(buf[k]), C.byref(ln[k]), C.byref(cap[k]))
                if rc != 0:
                    errs.append(lib.mgb_last_error())
                lib.mgb_get_stats(gi, C.byref(st))
                with cv:
                    for f in tot:
                        tot[f] += getattr(st, f)
                    done[k] = gcs
                    cv.notify_all()

        def writer():  # route A: the text in input order, as bench.py's writer makes it
            for k in range(M):
                with cv:
                    cv.wait_for(lambda: k in done or bool(errs))
                    if errs:
                        return
                    gcs = done.pop(k)
                lo, hi = mbs[k]
                t0 = time.perf_counter()
                lib.mgb_write_gaf_batch(g, hi - lo, gcs, sub(qlens, C.c_int, lo), sub(cnames, C.c_char_p, lo), mo.flag, gaf_threads,
                                        C.byref(buf[k]), C.byref(ln[k]), C.byref(cap[k]))
                lib.mgb_free_batch(hi - lo, gcs)
                writer_ms[0] += (time.perf_counter() - t0) * 1e3

        c0, t0 = cpu_s(), time.perf_counter()
        th = [threading.Thread(target=mapper) for _ in range(n_pipe)] + ([threading.Thread(target=writer)] if route == "A" else [])
        for t in th:
            t.start()
        for t in th:
            t.join()
        wall, cpu = (time.perf_counter() - t0) * 1e3, cpu_s() - c0
        assert not errs, errs
        h = hashlib.md5()
        for k in range(M):
            h.update(C.string_at(buf[k], ln[k].value))
        return wall, cpu, h.hexdigest(), tot, writer_ms[0]

    for _ in range(a.warmup):
        assert step("A")[2] == step("B")[2], "the routes' texts differ (warm-up)"
    res = {"A": [], "B": []}
    for s in range(a.steps):
        ra, rb = step("A"), step("B")
        assert ra[2] == rb[2], "step %d: the routes' texts differ (md5 %s vs %s)" % (s, ra[2], rb[2])
        res["A"].append(ra), res["B"].append(rb)
    gpu = gpu_info()
    text_bytes = sum(x.value for x in bufs["B"][1])
    lines = []
    for route, what in (("A", "mg_map_batch + mgb_write_gaf_batch + mgb_free_batch (objects, host writer)"),
                        ("B", "mgb_map_batch_gaf (text formatted on the device)")):
        rs = res[route]
        k = len(rs)
        wall = sum(r[0] for r in rs) / k
        lines.append({
            "route": route, "what": what, "workload": bench.workload_text(a.workload, n), "reads": n, "bases": bases,
            "mini_batches": M, "pipe": n_pipe, "host_threads": host_threads, "writer_threads": gaf_threads if route == "A" else 0,
            "steps": k, "warmup": a.warmup, "wall_ms_per_step": wall, "e2e_gbp_s": bases / (wall / 1e3) / 1e9,
            "host_cpu_s_per_step": sum(r[1] for r in rs) / k, "d2h_bytes_per_step": sum(r[3]["out_bytes"] for r in rs) / k,
            "t_dev_span_ms": sum(r[3]["t_dev_span_ms"] for r in rs) / k, "t_gaf_ms": sum(r[3]["t_gaf_ms"] for r in rs) / k,
            "t_asm_ms": sum(r[3]["t_asm_ms"] for r in rs) / k, "writer_ms": sum(r[4] for r in rs) / k,
            "n_launches_per_step": sum(r[3]["n_launches"] for r in rs) / k, "gaf_text_bytes": text_bytes,
            "text_md5_last_step": rs[-1][2], "text_identical": True, "gpu": gpu, "host_cores": ncores,
        })
    out = "".join(json.dumps(x) + "\n" for x in lines)
    sys.stdout.write(out)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out)
    for r in "AB":  # the text buffers are the caller's to free
        for b in bufs[r][0]:
            if b.value:
                C.CDLL(None).free(b)
    lib.mg_idx_destroy(gi)
    lib.mgb_gfa_destroy(g)
    lib.mgb_reads_free(rd)


if __name__ == "__main__":
    main()
