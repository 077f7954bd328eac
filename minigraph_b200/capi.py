"""ctypes view of include/mgb200.h -- the C ABI shared by libmgb200.so and the reference (minigraph.h).

The same structure definitions bind (a) the product library, (b) tests/hostsim and (c) oracle/_ref/libmgref.so,
because the ABI *is* the reference's (minigraph.h:41-176, gfa.h:33-106)."""
import ctypes as C
import os

MG_M_RMQ = 0x8000
MG_M_CIGAR = 0x4000000
MG_M_PRINT_2ND = 0x2000
MG_M_VERTEX_COOR = 0x800
MG_M_SHOW_UNMAP = 0x100000
MG_M_NO_COMP_PATH = 0x200000
MG_M_WRITE_LCHAIN = 0x800000
MG_M_WRITE_MZ = 0x1000000


class mg128_t(C.Structure):
    _fields_ = [("x", C.c_uint64), ("y", C.c_uint64)]


class mg_idxopt_t(C.Structure):
    _fields_ = [("w", C.c_int), ("k", C.c_int), ("bucket_bits", C.c_int)]


class mg_mapopt_t(C.Structure):  # minigraph.h:51-77
    _fields_ = [
        ("flag", C.c_uint64), ("mini_batch_size", C.c_int64), ("seed", C.c_int), ("max_qlen", C.c_int),
        ("pe_ori", C.c_int), ("occ_max1", C.c_int), ("occ_max1_cap", C.c_int), ("occ_max1_frac", C.c_float),
        ("bw", C.c_int), ("bw_long", C.c_int), ("rmq_size_cap", C.c_int), ("rmq_rescue_size", C.c_int),
        ("rmq_rescue_ratio", C.c_float), ("max_gap_pre", C.c_int), ("max_gap", C.c_int), ("max_gap_ref", C.c_int),
        ("max_frag_len", C.c_int), ("div", C.c_float), ("chn_pen_gap", C.c_float), ("chn_pen_skip", C.c_float),
        ("max_lc_skip", C.c_int), ("max_lc_iter", C.c_int), ("max_gc_skip", C.c_int), ("min_lc_cnt", C.c_int),
        ("min_lc_score", C.c_int), ("min_gc_cnt", C.c_int), ("min_gc_score", C.c_int), ("gdp_max_ed", C.c_int),
        ("lc_max_trim", C.c_int), ("lc_max_occ", C.c_int), ("mask_level", C.c_float), ("sub_diff", C.c_int),
        ("best_n", C.c_int), ("pri_ratio", C.c_float), ("ref_bonus", C.c_int), ("cap_kalloc", C.c_int64),
        ("min_cov_mapq", C.c_int), ("min_cov_blen", C.c_int),
    ]


class mg_idx_t(C.Structure):
    _fields_ = [("g", C.c_void_p), ("es", C.c_void_p), ("b", C.c_int32), ("w", C.c_int32), ("k", C.c_int32),
                ("flag", C.c_int32), ("n_seg", C.c_int32), ("B", C.c_void_p)]


class mg_llchain_t(C.Structure):
    _fields_ = [("off", C.c_int32), ("cnt", C.c_int32), ("v", C.c_uint32), ("score", C.c_int32), ("ed", C.c_int32)]


class mg_cigar_t(C.Structure):
    _fields_ = [("n_cigar", C.c_int32), ("mlen", C.c_int32), ("blen", C.c_int32), ("aplen", C.c_int32),
                ("ss", C.c_int32), ("ee", C.c_int32)]  # followed by uint64 cigar[]


class mg_ds_t(C.Structure):
    _fields_ = [("len", C.c_int32), ("n_off", C.c_int32), ("off", C.POINTER(C.c_int32)), ("ds", C.c_void_p)]


class mg_gchain_t(C.Structure):
    _fields_ = [
        ("id", C.c_int32), ("parent", C.c_int32), ("off", C.c_int32), ("cnt", C.c_int32), ("n_anchor", C.c_int32),
        ("score", C.c_int32), ("qs", C.c_int32), ("qe", C.c_int32), ("plen", C.c_int32), ("ps", C.c_int32),
        ("pe", C.c_int32), ("blen", C.c_int32), ("mlen", C.c_int32), ("div", C.c_float), ("hash", C.c_uint32),
        ("subsc", C.c_int32), ("n_sub", C.c_int32), ("mapq", C.c_uint32, 8), ("flt", C.c_uint32, 1),
        ("dummy", C.c_uint32, 23), ("p", C.POINTER(mg_cigar_t)), ("ds", mg_ds_t),
    ]


class mg_gchains_t(C.Structure):
    _fields_ = [("km", C.c_void_p), ("n_gc", C.c_int32), ("n_lc", C.c_int32), ("n_a", C.c_int32),
                ("rep_len", C.c_int32), ("gc", C.POINTER(mg_gchain_t)), ("lc", C.POINTER(mg_llchain_t)),
                ("a", C.POINTER(mg128_t))]


class gfa_seg_t(C.Structure):  # gfa.h:65-74
    _fields_ = [("len", C.c_int32), ("del_circ", C.c_uint32), ("snid", C.c_int32), ("soff", C.c_int32),
                ("rank", C.c_int32), ("name", C.c_char_p), ("seq", C.c_void_p), ("utg", C.c_void_p),
                ("aux_m", C.c_uint32), ("aux_l", C.c_uint32), ("aux", C.c_void_p)]


class gfa_sseq_t(C.Structure):
    _fields_ = [("name", C.c_char_p), ("min", C.c_int32), ("max", C.c_int32), ("rank", C.c_int32)]


class gfa_t(C.Structure):  # gfa.h:89-101
    _fields_ = [("m_seg", C.c_uint32), ("n_seg", C.c_uint32), ("max_rank", C.c_uint32), ("seg", C.POINTER(gfa_seg_t)),
                ("h_names", C.c_void_p), ("m_sseq", C.c_uint32), ("n_sseq", C.c_uint32),
                ("sseq", C.POINTER(gfa_sseq_t)), ("h_snames", C.c_void_p), ("m_arc", C.c_uint64),
                ("n_arc", C.c_uint64), ("arc", C.c_void_p), ("link_aux", C.c_void_p), ("idx", C.POINTER(C.c_uint64))]


class mgb_stats_t(C.Structure):
    _fields_ = [("t_h2d_ms", C.c_double), ("t_seed_ms", C.c_double), ("t_chain_ms", C.c_double),
                ("t_align_ms", C.c_double), ("t_d2h_ms", C.c_double), ("t_host_ms", C.c_double),
                ("t_wfa_ms", C.c_double), ("t_finish_ms", C.c_double), ("t_dev_span_ms", C.c_double), ("skip1_len", C.c_int64), ("skip2_len", C.c_int64), ("n_jobs_side", C.c_int64), ("n_slots", C.c_int64), ("t_pack_ms", C.c_double), ("t_asm_ms", C.c_double),
                ("n_jobs", C.c_int64), ("n_jobs_mid", C.c_int64), ("n_jobs_big", C.c_int64),
                ("n_reads", C.c_int64), ("n_bases", C.c_int64), ("n_seeds", C.c_int64), ("n_anchors_out", C.c_int64),
                ("n_chains_out", C.c_int64), ("n_minimizers", C.c_int64), ("out_bytes", C.c_int64),
                ("n_launches", C.c_int64), ("n_retry", C.c_int64), ("arena_peak", C.c_uint64), ("t_kernel_ms", C.c_double * 10), ("prof", C.c_uint64 * 32), ("t_lab_ms", C.c_double), ("n_lab_new", C.c_int64), ("n_lab_big", C.c_int64), ("h2d_bytes", C.c_int64),
                ("w_gpu_wait_ms", C.c_double), ("w_slot_wait_ms", C.c_double), ("w_upload_ms", C.c_double), ("w_pass_ms", C.c_double), ("w_redo_ms", C.c_double), ("w_download_ms", C.c_double),
                ("t_gaf_ms", C.c_double)]


class mgb_reads_t(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_bases", C.c_int64), ("name", C.POINTER(C.c_char_p)), ("seq", C.POINTER(C.c_char_p)),
                ("len", C.POINTER(C.c_int)), ("block", C.c_void_p)]


KERNEL_NAMES = ["k_seed", "k_chain", "k_gchain", "k_index_sketch", "k_wfa_small", "k_finish", "k_wfa_mid", "k_wfa_big", "k_gwfa", "k_gchain_gen"]
PROF_NAMES = ["wfa_fast_cyc", "wfa_fast_n", "wfa_slow_cyc", "wfa_slow_n", "wfa_max_cyc", "wfa_cells", "wfa_tb_cyc", "gc_dp_cyc", "gc_gen_cyc",
              "gc_post_cyc", "gc_plan_cyc", "fin_cigar_cyc", "fin_ds_cyc", "seed_sketch_cyc", "seed_match_cyc", "seed_sort_cyc", "chain_dp_cyc",
              "chain_onchip_n", "chain_rmq_cyc", "chain_post_cyc", "wfa_mid_cyc", "wfa_mid_n", "gc_gwfa_cyc", "gc_bridge_shortk_cyc", "gc_extra_sort_cyc", "gwfa_max_cyc", "gc_dp_max_cyc", "wfa_cta_cyc", "wfa_cta_n", "lab_cyc", "lab_n"]


def bind_mapping_api(lib):
    """Declare the prototypes of the symbols that exist in both the reference and libmgb200."""
    lib.mg_index.restype = C.POINTER(mg_idx_t)
    lib.mg_index.argtypes = [C.POINTER(gfa_t), C.POINTER(mg_idxopt_t), C.c_int, C.POINTER(mg_mapopt_t)]
    lib.mg_idx_destroy.restype = None
    lib.mg_idx_destroy.argtypes = [C.POINTER(mg_idx_t)]
    lib.mg_tbuf_init.restype = C.c_void_p
    lib.mg_tbuf_destroy.restype = None
    lib.mg_tbuf_destroy.argtypes = [C.c_void_p]
    lib.mg_map.restype = C.POINTER(mg_gchains_t)
    lib.mg_map.argtypes = [C.POINTER(mg_idx_t), C.c_int, C.c_char_p, C.c_void_p, C.POINTER(mg_mapopt_t), C.c_char_p]
    lib.mg_gchain_free.restype = None
    lib.mg_gchain_free.argtypes = [C.POINTER(mg_gchains_t)]
    lib.mg_idx_get.restype = C.POINTER(C.c_uint64)
    lib.mg_idx_get.argtypes = [C.POINTER(mg_idx_t), C.c_uint64, C.POINTER(C.c_int)]
    return lib


_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def env_params():
    """engine switches from the environment: MGB_PARAMS="wfa_v2=1,cta_len=1500" (pairs for mgb_set_param)"""
    out = {}
    for kv in os.environ.get("MGB_PARAMS", "").split(","):
        if "=" in kv:
            k, v = kv.split("=", 1)
            out[k.strip()] = int(v, 0)
    return out


def apply_env_params(lib):
    for k, v in env_params().items():
        if lib.mgb_set_param(k.encode(), v) != 0:
            raise RuntimeError("MGB_PARAMS: unknown engine parameter %r" % k)
    return lib


def load_product(path=None):
    """Load libmgb200.so (the CUDA build). Fails loudly when it has not been built -- there is no fallback."""
    path = path or os.environ.get("MGB_LIB") or os.path.join(_REPO, "minigraph_b200", "libmgb200.so")  # MGB_LIB: another build of the same library (A/B runs of bench.py)
    if not os.path.exists(path):
        raise RuntimeError("libmgb200.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    return apply_env_params(bind_engine_api(bind_mapping_api(lib)))


def bind_engine_api(lib):
    lib.mg_map_batch.restype = C.c_int
    lib.mg_map_batch.argtypes = [C.POINTER(mg_idx_t), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_char_p),
                                 C.POINTER(C.c_char_p), C.POINTER(C.POINTER(mg_gchains_t)), C.POINTER(mg_mapopt_t)]
    lib.mgb_last_error.restype = C.c_char_p
    lib.mgb_get_stats.restype = None
    lib.mgb_get_stats.argtypes = [C.POINTER(mg_idx_t), C.POINTER(mgb_stats_t)]
    lib.mgb_set_param.restype = C.c_int
    lib.mgb_set_param.argtypes = [C.c_char_p, C.c_int64]
    lib.mgb_gfa_read.restype = C.POINTER(gfa_t)
    lib.mgb_gfa_read.argtypes = [C.c_char_p]
    lib.mgb_gfa_destroy.restype = None
    lib.mgb_gfa_destroy.argtypes = [C.POINTER(gfa_t)]
    lib.mgb_write_gaf.restype = None
    lib.mgb_write_gaf.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(gfa_t),
                                  C.POINTER(mg_gchains_t), C.c_int32, C.c_char_p, C.c_uint64]
    lib.mgb_test_wfa.restype = C.c_int
    lib.mgb_test_wfa.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_uint32), C.c_int, C.POINTER(C.c_int)]
    lib.mg_map_batch_frag.restype = C.c_int
    lib.mg_map_batch_frag.argtypes = [C.POINTER(mg_idx_t), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                      C.POINTER(C.POINTER(mg_gchains_t)), C.POINTER(mg_mapopt_t)]
    lib.mgb_reads_load.restype = C.POINTER(mgb_reads_t)
    lib.mgb_reads_load.argtypes = [C.c_char_p, C.c_int64]
    lib.mgb_reads_free.restype = None
    lib.mgb_reads_free.argtypes = [C.POINTER(mgb_reads_t)]
    lib.mgb_free_batch.restype = None
    lib.mgb_free_batch.argtypes = [C.c_int, C.POINTER(C.POINTER(mg_gchains_t))]
    lib.mgb_write_gaf_batch.restype = None
    lib.mgb_write_gaf_batch.argtypes = [C.POINTER(gfa_t), C.c_int, C.POINTER(C.POINTER(mg_gchains_t)), C.POINTER(C.c_int),
                                        C.POINTER(C.c_char_p), C.c_uint64, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.mgb_map_batch_gaf.restype = C.c_int
    lib.mgb_map_batch_gaf.argtypes = [C.POINTER(mg_idx_t), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                      C.POINTER(mg_mapopt_t), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    return lib
