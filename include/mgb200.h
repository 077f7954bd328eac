/* mgb200.h -- C ABI of libmgb200.so, the B200-native replacement of minigraph's seed-chain-align hot path.
 *
 * The library is a drop-in for the mapping entry points of the reference: it keeps the symbol names, argument
 * meaning and ownership rules of minigraph.h so that the unmodified C host (main.c, gfa-*.c, bseq.c, format.c,
 * options.c, kthread.c ...) links against it.  Struct layouts below are binary compatible with the reference
 * headers they cite; they are restated here (not included) so that the library builds without the reference tree.
 * If the reference headers are included first (MINIGRAPH_H / __GFA_H__ defined), the restated types are skipped.
 *
 * Every entry point needs a CUDA device (sm_100a); there is no CPU fallback: without a device mg_index() returns
 * NULL after printing an error, and mgb_last_error() tells why.
 */
#ifndef MGB200_H
#define MGB200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------------------
 * Types restated from the reference (binary compatible)
 * ---------------------------------------------------------------------------------------------------------- */
#ifndef __GFA_H__
#define __GFA_H__ /* the restated declarations below stand in for gfa.h */
typedef struct { /* gfa.h:33-39 */
	uint64_t v_lv;
	uint32_t w;
	int32_t rank;
	int32_t ov, ow;
	uint64_t link_id:61, strong:1, del:1, comp:1;
} gfa_arc_t;

typedef struct { uint32_t m_aux, l_aux; uint8_t *aux; } gfa_aux_t; /* gfa.h:50-53 */

typedef struct gfa_utg_s gfa_utg_t; /* gfa.h:55-63, opaque here */

typedef struct { /* gfa.h:65-74 */
	int32_t len;
	uint32_t del:16, circ:16;
	int32_t snid;
	int32_t soff;
	int32_t rank;
	char *name, *seq;
	gfa_utg_t *utg;
	gfa_aux_t aux;
} gfa_seg_t;

typedef struct { char *name; int32_t min, max, rank; } gfa_sseq_t; /* gfa.h:82-85 */

typedef struct { /* gfa.h:89-101 */
	uint32_t m_seg, n_seg, max_rank;
	gfa_seg_t *seg;
	void *h_names;
	uint32_t m_sseq, n_sseq;
	gfa_sseq_t *sseq;
	void *h_snames;
	uint64_t m_arc, n_arc;
	gfa_arc_t *arc;
	gfa_aux_t *link_aux;
	uint64_t *idx;
} gfa_t;

typedef struct { const char *seq; int32_t len; } gfa_edseq_t; /* gfa.h:103-106 */
#endif

#ifndef MINIGRAPH_H
#define MINIGRAPH_H /* the restated declarations below stand in for minigraph.h */
#define MG_M_RMQ    0x8000      /* minigraph.h:24 */
#define MG_M_CIGAR  0x4000000   /* minigraph.h:35 */

typedef struct { uint64_t x, y; } mg128_t; /* minigraph.h:41 */

typedef struct { int w, k; int bucket_bits; } mg_idxopt_t; /* minigraph.h:46-49 */

typedef struct { /* minigraph.h:51-77 */
	uint64_t flag;
	int64_t mini_batch_size;
	int seed;
	int max_qlen;
	int pe_ori;
	int occ_max1, occ_max1_cap;
	float occ_max1_frac;
	int bw, bw_long;
	int rmq_size_cap;
	int rmq_rescue_size;
	float rmq_rescue_ratio;
	int max_gap_pre, max_gap, max_gap_ref, max_frag_len;
	float div;
	float chn_pen_gap, chn_pen_skip;
	int max_lc_skip, max_lc_iter, max_gc_skip;
	int min_lc_cnt, min_lc_score;
	int min_gc_cnt, min_gc_score;
	int gdp_max_ed, lc_max_trim, lc_max_occ;
	float mask_level;
	int sub_diff;
	int best_n;
	float pri_ratio;
	int ref_bonus;
	int64_t cap_kalloc;
	int min_cov_mapq, min_cov_blen;
} mg_mapopt_t;

typedef struct { /* minigraph.h:93-98 */
	const gfa_t *g;
	gfa_edseq_t *es;
	int32_t b, w, k, flag, n_seg;
	struct mg_idx_bucket_s *B; /* hidden: here it points to the engine's model (host copy + device image) */
} mg_idx_t;

typedef struct { int32_t off, cnt; uint32_t v; int32_t score; int32_t ed; } mg_llchain_t; /* minigraph.h:108-113 */

typedef struct { /* minigraph.h:115-118 */
	int32_t n_cigar, mlen, blen, aplen, ss, ee;
	uint64_t cigar[];
} mg_cigar_t;

typedef struct { int32_t len, n_off, *off; char *ds; } mg_ds_t; /* minigraph.h:120-123 */

typedef struct { /* minigraph.h:125-138 */
	int32_t id, parent;
	int32_t off, cnt;
	int32_t n_anchor, score;
	int32_t qs, qe;
	int32_t plen, ps, pe;
	int32_t blen, mlen;
	float div;
	uint32_t hash;
	int32_t subsc, n_sub;
	uint32_t mapq:8, flt:1, dummy:23;
	mg_cigar_t *p;
	mg_ds_t ds;
} mg_gchain_t;

typedef struct { /* minigraph.h:140-146 */
	void *km;
	int32_t n_gc, n_lc, n_a, rep_len;
	mg_gchain_t *gc;
	mg_llchain_t *lc;
	mg128_t *a;
} mg_gchains_t;

typedef struct mg_tbuf_s mg_tbuf_t; /* minigraph.h:148, opaque */
#endif

/* ------------------------------------------------------------------------------------------------------------
 * Entry points that replace reference symbols one to one
 * ---------------------------------------------------------------------------------------------------------- */

/* replaces index.c:211-230 mg_index(): upper-cases the segments of g (index.c:215-220), returns NULL when the graph
 * has overlapping links (index.c:192-196), builds the minimizer index, uploads graph+index to the GPU and updates
 * mo->occ_max1 / lc_max_occ / bw_long exactly like options.c:120-134 mg_opt_update(). n_threads is ignored.
 * The GPU is the engine parameter "device" (default 0); with the environment variable MGB_DEVICES ("0-7", "0,2,5") the index is
 * replicated on every listed GPU and each mg_map_batch*() call is cut into one contiguous part per GPU (results in input order).
 * Returns NULL on failure (no CUDA device, out of device memory, overlapping links) with the reason in mgb_last_error(). */
mg_idx_t *mg_index(gfa_t *g, const mg_idxopt_t *io, int n_threads, mg_mapopt_t *mo);

/* replaces index.c:30-46 mg_idx_destroy() */
void mg_idx_destroy(mg_idx_t *gi);

/* replaces index.c:67-72 mg_idx_get(): host view of one occurrence list (ascending seg<<32|pos<<1|strand) */
const uint64_t *mg_idx_get(const mg_idx_t *gi, uint64_t minier, int *n);

/* replaces index.c:74-93 mg_idx_cal_quantile() */
void mg_idx_cal_quantile(const mg_idx_t *gi, int32_t m, float f[], int32_t q[]);

/* replaces index.c:108-113 mg_idx_hfree(): the one other index.c symbol the remaining host files reference
 * (shortk.c:191, always with a NULL handle); a no-op here */
void mg_idx_hfree(void *h);

/* replace map-algo.c:14-27 mg_tbuf_init()/mg_tbuf_destroy(): the per-thread arena becomes a handle without state */
mg_tbuf_t *mg_tbuf_init(void);
void mg_tbuf_destroy(mg_tbuf_t *b);

/* replaces map-algo.c:340-495 mg_map_frag(): gcs[0] receives a malloc()ed result owned by the caller (free with
 * mg_gchain_free), or NULL when the fragment is empty, has more than 255 segments or is longer than opt->max_qlen
 * (map-algo.c:359-360); gcs[i>0] = NULL. With n_segs > 1 the concatenated fragment is mapped and no CIGAR is produced
 * (map-algo.c:34-45,464,475). One fragment per launch: correct but slow -- use mg_map_batch for single-segment reads.
 * Re-entrancy: like the reference's (which needs one mg_tbuf_t per thread, map-algo.c:9-12), any number of host threads may call
 * mg_map_frag()/mg_map()/mg_map_batch*() on one mg_idx_t at the same time.  Every call in flight owns a "slot" (stream, staging
 * buffers, pools, worker arenas); at most "slots" calls (engine parameter, default 3) run at once, further callers wait.
 * This entry point has no error return (the reference's has none): an internal failure ends the process as an assert would. */
void mg_map_frag(const mg_idx_t *gi, int n_segs, const int *qlens, const char **seqs, mg_gchains_t **gcs, mg_tbuf_t *b, const mg_mapopt_t *opt, const char *qname);

/* replaces map-algo.c:497-502 mg_map() */
mg_gchains_t *mg_map(const mg_idx_t *gi, int qlen, const char *seq, mg_tbuf_t *b, const mg_mapopt_t *opt, const char *qname);

/* replaces gchain1.c:522-535 mg_gchain_free() (results are plain malloc/calloc blocks, km == NULL) */
void mg_gchain_free(mg_gchains_t *gs);

/* ------------------------------------------------------------------------------------------------------------
 * New entry point: the GPU batch dispatcher that replaces kt_for(worker_for) at gmap.c:99
 * ---------------------------------------------------------------------------------------------------------- */

/* Map n_reads single-segment reads in one go. seqs[i] must be upper-case (gmap.c:81) and need not be 0-terminated;
 * names[i] may be NULL. gcs[i] is filled exactly as worker_for() (gmap.c:29-64) would fill s->gcs[off].
 * Returns 0, or a negative code after printing the reason (no partial results are left behind; a CUDA failure -- out of memory,
 * a fault -- is reported this way too, the library never ends the process from here).  A host that maps mini-batch i+1 from a
 * second thread while the first is still inside the call for mini-batch i overlaps packing, copies and result assembly of one
 * with the kernels of the other, as the reference's kt_pipeline overlaps its steps (gmap.c:176-177). */
int mg_map_batch(const mg_idx_t *gi, int n_reads, const int *qlens, const char *const *seqs, const char *const *names,
				 mg_gchains_t **gcs, const mg_mapopt_t *opt);

/* The same for fragments of several segments (read pairs, the `sr` preset): fragment f owns n_seg[f] consecutive entries of
 * qlens/seqs/gcs; the result of the concatenated fragment goes to its first gcs entry, the others are NULL -- what
 * worker_for() leaves without MG_M_INDEPEND_SEG (gmap.c:46-48). names[] is per fragment. The caller reverse-complements
 * mates beforehand as gmap.c:38-40 does. */
int mg_map_batch_frag(const mg_idx_t *gi, int n_frag, const int *n_seg, const int *qlens, const char *const *seqs, const char *const *names,
					  mg_gchains_t **gcs, const mg_mapopt_t *opt);

/* mg_gchain_free() over a whole batch (what step 2 of the reference pipeline does read by read, gmap.c:130); entries are set to NULL */
void mgb_free_batch(int n_reads, mg_gchains_t **gcs);

/* Map n_reads single-segment reads and return their GAF text, formatted on the device: byte for byte what
 * mg_map_batch(gi, n_reads, qlens, seqs, names, gcs, opt) followed by
 * mgb_write_gaf_batch(gi->g, n_reads, gcs, qlens, names, opt->flag, ...) produces, for every flag bit mgb_write_gaf() handles
 * except MG_M_WRITE_LCHAIN / MG_M_WRITE_MZ (-S, --write-mz), which are refused with a negative code.  The flags are opt->flag,
 * as the reference passes them to mg_write_gaf (gmap.c); a NULL names or names[i] prints as "*".
 * (*out, *out_len, *out_cap) as in mgb_write_gaf_batch(). Returns 0, or a negative code with the reason in mgb_last_error();
 * on failure *out_len is 0 and no text is left behind.
 * The call follows the rules of mg_map_batch(): slots and concurrent callers, MGB_DEVICES (the text comes back in input order),
 * the large-arena retry pass, growth of overflowing pools, error reporting.  No mg_gchains_t is built: the text is formatted
 * from the device's result blobs, and only the text (plus 16 bytes per record for the dv:f field, which the host prints because
 * its value comes from the host's libm) crosses PCIe.  The graph's names go to the device at the first call on an index. */
int mgb_map_batch_gaf(const mg_idx_t *gi, int n_reads, const int *qlens, const char *const *seqs, const char *const *names,
                      const mg_mapopt_t *opt, char **out, size_t *out_len, size_t *out_cap);

/* ------------------------------------------------------------------------------------------------------------
 * Engine controls and instrumentation (not part of the reference API)
 * ---------------------------------------------------------------------------------------------------------- */

typedef struct {
	double t_h2d_ms, t_seed_ms, t_chain_ms, t_align_ms, t_d2h_ms, t_host_ms; /* last batch, CUDA events / host clock */
	double t_wfa_ms, t_finish_ms; /* t_align_ms = graph chaining + alignment plan; t_wfa_ms = gap alignment jobs; t_finish_ms = cigar/ds/blob */
	double t_dev_span_ms;   /* device time from the first kernel start to the last kernel end over all sub-batches (they overlap) */
	int64_t skip1_len, skip2_len; /* WFA tier routing this batch ran with: gaps at or above these lengths skipped tier 1 / tier 2 */
	int64_t n_jobs_side;    /* gaps aligned by the tier-3 launch that runs beside tiers 1/2 */
	int64_t n_slots;        /* sub-batches the batch was cut into (each on its own stream and host thread) */
	double t_pack_ms, t_asm_ms; /* host: packing reads into the staging buffer; building mg_gchains_t objects (mgb_map_batch_gaf: inserting dv:f and copying the text to the caller) */
	int64_t n_jobs;         /* WFA jobs of the batch */
	int64_t n_jobs_mid, n_jobs_big; /* jobs that went to tier 2 / tier 3 */
	int64_t n_reads, n_bases;
	int64_t n_seeds;        /* sum of seeds entering the chaining kernel */
	int64_t n_anchors_out;  /* sum of anchors kept in linear chains */
	int64_t n_chains_out;   /* sum of linear chains out of the DP */
	int64_t n_minimizers;
	int64_t out_bytes;      /* result bytes copied back (mgb_map_batch_gaf: the text and its dv:f fix-up records) */
	int64_t n_launches;     /* kernels launched for the batch (mgb_map_batch_gaf: one more, k_gaf_size + scan + k_gaf_write in place of the two blob kernels) */
	int64_t n_retry;        /* reads re-run with a larger arena */
	uint64_t arena_peak;    /* largest per-worker arena use */
	double t_kernel_ms[10]; /* CUDA-event time of each kernel of the first pass: k_seed, k_chain, k_gchain, (index), k_wfa_small, k_finish, k_wfa_mid, k_wfa_big, k_gwfa, k_gchain_gen */
	uint64_t prof[32];      /* device cycle counters per phase (see mgb_pipeline.cuh PROF_*) */
	double t_lab_ms;        /* k_gc_labels: reachability labels of source vertices seen for the first time (0 once the table is warm) */
	int64_t n_lab_new;      /* such sources in this batch */
	int64_t n_lab_big;      /* ... of which needed the second, warp-per-source pass */
	int64_t h2d_bytes;      /* bytes of reads and per-read tables copied to the device (reads travel 2 bits per base unless they hold letters other than A/C/G/T) */
	double w_gpu_wait_ms;   /* host wall clock spent waiting for the kernels of another call in flight to finish */
	double w_slot_wait_ms, w_upload_ms, w_pass_ms, w_redo_ms, w_download_ms; /* host wall clock of the call: waiting for a slot; packing + H2D; the kernels of the first pass
	                           with the host syncs between them; the large-arena pass over reads that outgrew their arena; result packing + D2H up to the assembly */
	double t_gaf_ms;        /* mgb_map_batch_gaf: CUDA-event time of the GAF kernels (k_gaf_size with its scan, k_gaf_write); 0 for mg_map_batch */
} mgb_stats_t;

/* test hook: align one gap through the tier-3 WFA path (exact up to max_iter cells, then the reference's chaining
 * heuristic, miniwfa.c:824-834, with checkpoints every `step` scores); returns n_cigar (len<<4|op) or a negative code */
int mgb_test_wfa(const char *ts, int tl, const char *qs, int ql, int64_t max_iter, int step, uint32_t *cigar, int cap, int *score);

const char *mgb_last_error(void);
void mgb_get_stats(const mg_idx_t *gi, mgb_stats_t *st);
/* knobs: "arena_mb" (per worker), "workers_per_sm", "device"; returns 0 if the key is known */
int mgb_set_param(const char *key, int64_t value);
const char *mgb_version(void);

/* Convenience for callers without a gfa_t (bench, tests): parse GFA/rGFA text the way gfa-io.c:294-337 gfa_read()
 * does for S/L lines with SN/SO/SR tags and plain FASTA, and finalize arcs like gfa-base.c:421-430. */
gfa_t *mgb_gfa_read(const char *fn);
void mgb_gfa_destroy(gfa_t *g);

/* Input side for hosts without the reference's bseq.c: a whole FASTA/FASTQ file (plain or gzip, "-" = stdin) parsed by kseq.h's rules
 * (bseq.c:46-98) and upper-cased (gmap.c:81) into the arrays mg_map_batch() takes.  max_bases > 0 stops after the record that
 * reaches it (the reference's mini-batch rule, bseq.c:70-72).  NULL if the file cannot be opened. */
typedef struct { int64_t n_reads, n_bases; const char **name, **seq; int *len; char *block; } mgb_reads_t;
mgb_reads_t *mgb_reads_load(const char *fn, int64_t max_bases);
void mgb_reads_free(mgb_reads_t *r);

/* Byte-exact GAF line(s) for one read, restating format.c:121-291 mg_write_gaf() for flag bits used by -c. The text is
 * appended to *buf (realloc()ed; *len and *cap updated). */
void mgb_write_gaf(char **buf, size_t *len, size_t *cap, const gfa_t *g, const mg_gchains_t *gs, int32_t qlen, const char *qname, uint64_t flag);

/* The same for a whole batch, input order preserved, formatted by n_threads host threads (0: up to 16). The text is
 * 0-terminated and *out_len receives its length. out_cap == NULL: *out is a fresh malloc() block the caller frees.
 * out_cap != NULL: (*out, *out_cap) is a buffer owned by the caller (NULL/0 the first time) that is reused and grown
 * with realloc semantics, like mgb_write_gaf() does with (buf, cap). */
void mgb_write_gaf_batch(const gfa_t *g, int n_reads, mg_gchains_t *const *gcs, const int *qlens, const char *const *names,
						 uint64_t flag, int n_threads, char **out, size_t *out_len, size_t *out_cap);

#ifdef __cplusplus
}
#endif
#endif
