// mgb_gaf.cuh -- the GAF text of a read, formatted on the device (mgb_map_batch_gaf).
//
// gaf_read() restates mgb_write_gaf() (mgb_gfa.cpp, itself a restatement of format.c:121-251) for one read, from the result
// blobs the kernels left in the output pool (ReadOut / GChain offsets), entered by all lanes of a warp.  It runs twice per read:
// k_gaf_size counts the bytes and the fix-up records, k_gaf_write writes them at the read's place after the exclusive scan.
// Both passes run the same code, so the sizes cannot disagree with the text.
//
// What the device does not print: `dv:f`.  div is (float)(log(ratio) / q_span) evaluated by the host's libm, which the device
// cannot reproduce bit for bit (SURVEY H3).  Every printed record leaves a GafFix instead, and the host inserts the field at that
// byte while it copies the text to the caller (gaf_div() and mgb_dv_text() hold the two rules).
#pragma once
#include "mgb_galign.cuh"

namespace mgb {

static const uint64_t F_VERTEX_COOR = 0x800, F_PRINT_2ND = 0x2000, F_SHOW_UNMAP = 0x100000, F_NO_COMP_PATH = 0x200000;
static const uint64_t F_WRITE_LCHAIN = 0x800000, F_WRITE_MZ = 0x1000000;

// the `dv:f` field of one printed record: inserted by the host at byte `at` of the read's text
struct GafFix { uint32_t at; int32_t n_mini, n_anchor, q_span; };
// the field's text, as mgb_write_gaf() prints it (mgb_gfa.cpp)
int gaf_dv_text(float div, char *b);

// Everything the GAF kernels read besides the pipeline's own arrays.  Names are kept without terminator: name i is
// blob[off[i] .. off[i+1]).
struct GafCtx {
	// the graph, uploaded once per model (gfa_seg_t / gfa_sseq_t fields the writer reads; segment lengths are GraphDev::seg_len)
	const char *seg_name; const uint64_t *seg_name_off; // [n_seg + 1]
	const int32_t *seg_snid, *seg_soff;
	const char *ss_name; const uint64_t *ss_name_off;   // [n_sseq + 1]
	const int32_t *ss_rank, *ss_min, *ss_max;
	const unsigned char *comp;                          // [256] the engine's comp_tab (gfa_comp_table)
	// the batch
	const char *rname; const uint64_t *rname_off;       // [n_reads + 1]; a NULL name travels as "*"
	uint64_t flag;                                      // the mapping flags (mg_mapopt_t::flag)
	uint64_t *text_off;                                 // [n_reads + 1]: bytes per read after k_gaf_size, offsets after the scan
	uint64_t *fix_off;                                  // [n_reads + 1]: fix-up records per read, the same way
	char *text;                                         // k_gaf_write: the text of the sub-batch
	GafFix *fix;                                        // k_gaf_write: its fix-up records
};

// The output of one read.  Every lane holds the same count; scalar bytes are stored by lane 0, runs of bytes by all lanes.
// d == NULL: count only.
struct GafOut {
	char *d;
	uint64_t n;
	int lane;
	MG_HD void put(char c) { if (d && lane == 0) d[n] = c; ++n; }
	MG_HD void putn(const char *s, uint64_t l) { if (d) for (uint64_t i = (uint64_t)lane; i < l; i += MGB_W) d[n + i] = s[i]; n += l; }
	MG_HD void puts(const char *s) { while (*s) put(*s++); }
	MG_HD void putd(int32_t c) // reference: format.c mg_sprintf_lite %d
	{
		char b[12];
		int l = 0;
		uint32_t x = c >= 0? (uint32_t)c : (uint32_t)0 - (uint32_t)c;
		do { b[l++] = (char)(x % 10 + '0'); x /= 10; } while (x > 0);
		if (c < 0) b[l++] = '-';
		while (l > 0) put(b[--l]);
	}
};

MG_HD inline int gaf_ndigits(uint32_t x) { int l = 1; while (x >= 10) x /= 10, ++l; return l; }

MG_HD inline void gaf_name(GafOut &o, const char *blob, const uint64_t *off, int64_t i) { o.putn(blob + off[i], off[i + 1] - off[i]); }

// ">sname:st-en" (format.c s_seg)
MG_HD inline void gaf_sseg(GafOut &o, const GafCtx &x, int rev, int32_t snid, int32_t st, int32_t en)
{
	o.put("><"[rev]); gaf_name(o, x.ss_name, x.ss_name_off, snid); o.put(':'); o.putd(st); o.put('-'); o.putd(en);
}

// The CIGAR, one op per lane: digits of the lengths placed by a warp prefix sum
MG_HD inline void gaf_cigar(GafOut &o, const uint64_t *cig, int32_t n_cigar, int rev)
{
	for (int32_t base = 0; base < n_cigar; base += MGB_W) {
		const int32_t j = base + o.lane;
		uint64_t c = 0;
		int32_t len = 0;
		if (j < n_cigar) c = cig[rev? n_cigar - 1 - j : j], len = gaf_ndigits((uint32_t)(c >> 4)) + 1;
		const int32_t end = warp_incl_scan_i32(len, o.lane), tot = warp_sum_i32(len);
		if (o.d && j < n_cigar) {
			char *p = o.d + o.n + (end - len);
			uint32_t v = (uint32_t)(c >> 4);
			for (int32_t k = len - 2; k >= 0; --k) p[k] = (char)(v % 10 + '0'), v /= 10;
			p[len - 1] = "MIDNSHP=XB"[c & 0xf];
		}
		o.n += (uint64_t)tot;
	}
}

// The ds string read backwards (format.c:226-246), one op per lane: op k of the input has the same length in the output and starts
// there at ds_len - end(k); ':' runs keep their order, '*' pairs are complemented, other ops are reversed and complemented with
// '[' and ']' swapped.
MG_HD inline void gaf_ds_rev(GafOut &o, const char *ds, int32_t ds_len, const int32_t *dof, int32_t n_off, const unsigned char *comp)
{
	if (n_off <= 0) return;
	if (o.d)
		for (int32_t k = o.lane; k < n_off; k += MGB_W) {
			const int32_t off = dof[k], en = k < n_off - 1? dof[k + 1] : ds_len;
			char *p = o.d + o.n + (ds_len - en);
			const char op = ds[off];
			*p++ = op;
			if (op == ':') for (int32_t j = off + 1; j < en; ++j) *p++ = ds[j];
			else if (op == '*') for (int32_t j = off + 1; j < en; ++j) *p++ = (char)comp[(uint8_t)ds[j]];
			else
				for (int32_t j = en - 1; j >= off + 1; --j)
					*p++ = ds[j] == '['? ']' : ds[j] == ']'? '[' : (char)comp[(uint8_t)ds[j]];
		}
	o.n += (uint64_t)(ds_len - dof[0]);
}

// The GAF lines of read r.  fix: where the write pass puts the read's fix-up records (NULL: count them into *n_fix only).
MG_HD inline void gaf_read(const GafCtx &x, const PipeCtx &c, const ReadOut &ro, int r, GafOut &o, GafFix *fix, uint32_t *n_fix)
{
	const uint64_t flag = x.flag;
	const int32_t qlen = c.b.seq_len[r];
	*n_fix = 0;
	if (ro.status != 0 || ro.n_gc <= 0) { // no result object, or one without chains
		if (flag & F_SHOW_UNMAP) { gaf_name(o, x.rname, x.rname_off, r); o.put('\t'); o.putd(qlen); o.puts("\t0\t0\t*\t*\t0\t0\t0\t0\t0\t0\n"); }
		return;
	}
	const char *blob = c.out + ro.blob_off;
	const GChain *gcs = (const GChain*)blob;
	const LLChain *lcs = (const LLChain*)(blob + align8((uint64_t)ro.n_gc * sizeof(GChain)));
	const GraphDev &g = c.g;
	int rev_sign = 0; // sticky across the records of one read, like the reference (format.c:123)
	for (int32_t i = 0; i < ro.n_gc; ++i) {
		const GChain *p = &gcs[i];
		if (p->id != p->parent && !(flag & F_PRINT_2ND)) continue;
		if (p->cnt == 0) continue;
		gaf_name(o, x.rname, x.rname_off, r);
		o.put('\t'); o.putd(qlen); o.put('\t'); o.putd(p->qs); o.put('\t'); o.putd(p->qe); o.puts("\t+\t");
		const uint64_t sign_pos = o.n - 2;
		int compact;
		if (flag & F_VERTEX_COOR) {
			compact = 0;
			for (int32_t j = 0; j < p->cnt; ++j) {
				const uint32_t v = lcs[p->off + j].v;
				o.put("><"[v & 1]); gaf_name(o, x.seg_name, x.seg_name_off, v >> 1);
			}
		} else { // stable-coordinate runs (format.c:141-177)
			int32_t last_pnid = -1, st = -1, en = -1, rev = -1;
			compact = flag & F_NO_COMP_PATH? 0 : 1;
			for (int32_t j = 0; j < p->cnt; ++j) {
				const uint32_t v = lcs[p->off + j].v, s = v >> 1;
				const int32_t snid = x.seg_snid[s], soff = x.seg_soff[s], slen = g.seg_len[s];
				if (snid < 0) {
					compact = 0;
					if (last_pnid >= 0) gaf_sseg(o, x, rev, last_pnid, st, en);
					last_pnid = -1, st = -1, en = -1, rev = -1;
					o.put("><"[v & 1]); gaf_name(o, x.seg_name, x.seg_name_off, s);
				} else {
					int cont = 0;
					if (last_pnid >= 0 && snid == last_pnid && (int32_t)(v & 1) == rev) {
						if (!(v & 1)) { if (soff == en) en = soff + slen, cont = 1; }
						else { if (soff + slen == st) st = soff, cont = 1; }
					}
					if (cont == 0) {
						if (last_pnid >= 0) compact = 0, gaf_sseg(o, x, rev, last_pnid, st, en);
						last_pnid = snid, rev = (int32_t)(v & 1), st = soff, en = st + slen;
					}
				}
			}
			if (last_pnid >= 0) {
				if (x.ss_rank[last_pnid] != 0 || x.ss_min[last_pnid] != 0) compact = 0;
				if (!compact) gaf_sseg(o, x, rev, last_pnid, st, en);
			} else compact = 0;
		}
		if (compact) {
			const int rev = (int)(lcs[p->off].v & 1);
			const uint32_t s = lcs[rev? p->off + p->cnt - 1 : p->off].v >> 1;
			const int32_t snid = x.seg_snid[s], soff = x.seg_soff[s];
			gaf_name(o, x.ss_name, x.ss_name_off, snid); o.put('\t'); o.putd(x.ss_max[snid]); o.put('\t');
			if (rev) {
				rev_sign = 1;
				if (o.d && o.lane == 0) o.d[sign_pos] = '-';
				o.putd(soff + (p->plen - p->pe)); o.put('\t'); o.putd(soff + (p->plen - p->ps));
			} else {
				o.putd(soff + p->ps); o.put('\t'); o.putd(soff + p->pe);
			}
		} else { o.put('\t'); o.putd(p->plen); o.put('\t'); o.putd(p->ps); o.put('\t'); o.putd(p->pe); }
		o.put('\t'); o.putd(p->has_cigar? p->c_mlen : p->mlen); o.put('\t'); o.putd(p->has_cigar? p->c_blen : p->blen);
		o.put('\t'); o.putd(p->mapq & 0xff); // (mg_gchain_t::mapq is an 8-bit field)
		o.puts("\ttp:A:"); o.put(p->id == p->parent? 'P' : 'S');
		if (p->has_cigar) { o.puts("\tNM:i:"); o.putd(p->c_blen - p->c_mlen); }
		o.puts("\tcm:i:"); o.putd(p->n_anchor); o.puts("\ts1:i:"); o.putd(p->score); o.puts("\ts2:i:"); o.putd(p->subsc);
		if (fix && o.lane == 0) { GafFix &f = fix[*n_fix]; f.at = (uint32_t)o.n, f.n_mini = p->n_mini, f.n_anchor = p->n_anchor, f.q_span = p->q_span; }
		++*n_fix;
		if (p->has_cigar) {
			o.puts("\tcg:Z:");
			gaf_cigar(o, (const uint64_t*)(c.out + p->cigar_off), p->n_cigar, rev_sign);
			o.puts("\tds:Z:");
			const char *ds = c.out + p->ds_off;
			if (rev_sign) gaf_ds_rev(o, ds, p->ds_len, (const int32_t*)(c.out + p->dsoff_off), p->n_dsoff, x.comp);
			else o.putn(ds, (uint64_t)p->ds_len);
		}
		o.put('\n');
	}
}

// k_gaf_size: the bytes and fix-up records of read r
MG_HD inline int stage_gaf_size(const GafCtx &x, const PipeCtx &c, const ReadOut *routs, int r, int lane)
{
	GafOut o = {0, 0, lane};
	uint32_t n_fix = 0;
	gaf_read(x, c, routs[r], r, o, 0, &n_fix);
	if (lane == 0) x.text_off[r] = o.n, x.fix_off[r] = n_fix;
	return 0;
}

// k_gaf_write: the text and fix-up records of read r at their place
MG_HD inline int stage_gaf_write(const GafCtx &x, const PipeCtx &c, const ReadOut *routs, int r, int lane)
{
	GafOut o = {x.text + x.text_off[r], 0, lane};
	uint32_t n_fix = 0;
	gaf_read(x, c, routs[r], r, o, x.fix + x.fix_off[r], &n_fix);
	return 0;
}

} // namespace mgb
