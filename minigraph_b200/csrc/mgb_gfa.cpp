// mgb_gfa.cpp -- host-side graph loader and GAF text writer of libmgb200 (pure C++, no CUDA).
//
//   mgb_gfa_read()   builds a gfa_t that is binary compatible with the reference's (gfa.h:89-101) from rGFA/GFA S/L lines or
//                    plain FASTA, and finalizes the arc array with the same sequence of sorts as gfa-base.c:421-430
//                    gfa_finalize(): the relative order of arcs leaving one vertex is decided by klib's *unstable* radix
//                    sort and is consumed by the graph walks on the device (SURVEY H10b), so the sort is replayed exactly.
//   mgb_write_gaf()  restates format.c:121-291 mg_write_gaf() byte for byte (rows (f)1 of SURVEY section 8).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ctype.h>
#include <math.h>
#include <zlib.h>
#include <string>
#include <vector>
#include <unordered_map>

#include "../../include/mgb200.h"
#include "mgb_common.cuh"

namespace {

typedef std::unordered_map<std::string, uint32_t> name_map_t;

struct KeyArc { uint64_t operator()(const gfa_arc_t &a) const { return a.v_lv; } };

void arc_sort(gfa_t *g) // reference: gfa-base.c:175-178 (radix_sort_arc, key v_lv, 8 bytes)
{
	std::vector<char> scratch((size_t)(g->n_arc / 64 + 512) * sizeof(mgb::RsRange) + 4096);
	mgb::Arena A;
	mgb::arena_init(A, scratch.data(), scratch.size());
	int rc = mgb::radix_sort_exact(A, g->arc, (int64_t)g->n_arc, 8, KeyArc());
	if (rc < 0) { fprintf(stderr, "[E::mgb200] arc sort failed\n"); abort(); }
}

bool arc_is_sorted(const gfa_t *g)
{
	for (uint64_t e = 1; e < g->n_arc; ++e)
		if (g->arc[e-1].v_lv > g->arc[e].v_lv) return false;
	return true;
}

void arc_index(gfa_t *g) // reference: gfa-base.c:180-195
{
	free(g->idx);
	g->idx = (uint64_t*)calloc((size_t)g->n_seg * 2 + 1, 8);
	uint64_t n = g->n_arc, last = 0;
	for (uint64_t i = 1; i <= n; ++i)
		if (i == n || (uint32_t)(g->arc[i-1].v_lv >> 32) != (uint32_t)(g->arc[i].v_lv >> 32))
			g->idx[(uint32_t)(g->arc[i-1].v_lv >> 32)] = last << 32 | (i - last), last = i;
}

int32_t add_seg(gfa_t *g, const char *name) // reference: gfa-base.c:77-98
{
	name_map_t *h = (name_map_t*)g->h_names;
	auto it = h->find(name);
	if (it != h->end()) return (int32_t)it->second;
	if (g->n_seg == g->m_seg) {
		uint32_t old_m = g->m_seg;
		g->m_seg = g->m_seg? g->m_seg << 1 : 16;
		g->seg = (gfa_seg_t*)realloc(g->seg, g->m_seg * sizeof(gfa_seg_t));
		memset(&g->seg[old_m], 0, (g->m_seg - old_m) * sizeof(gfa_seg_t));
	}
	gfa_seg_t *s = &g->seg[g->n_seg++];
	s->name = strdup(name);
	s->del = 0, s->len = 0;
	s->snid = s->soff = s->rank = -1;
	(*h)[name] = g->n_seg - 1;
	return (int32_t)g->n_seg - 1;
}

int32_t sseq_add(gfa_t *g, const char *sname) // reference: gfa-base.c:100-115
{
	name_map_t *h = (name_map_t*)g->h_snames;
	auto it = h->find(sname);
	if (it != h->end()) return (int32_t)it->second;
	if (g->n_sseq == g->m_sseq) {
		g->m_sseq = g->m_sseq? g->m_sseq + (g->m_sseq >> 1) : 16;
		g->sseq = (gfa_sseq_t*)realloc(g->sseq, g->m_sseq * sizeof(gfa_sseq_t));
	}
	gfa_sseq_t *ss = &g->sseq[g->n_sseq++];
	ss->name = strdup(sname);
	ss->min = -1, ss->max = -1, ss->rank = -1;
	(*h)[sname] = g->n_sseq - 1;
	return (int32_t)g->n_sseq - 1;
}

void sseq_update(gfa_t *g, const gfa_seg_t *s) // reference: gfa-base.c:126-138
{
	if (s->snid < 0 || (uint32_t)s->snid >= g->n_sseq) return;
	gfa_sseq_t *ps = &g->sseq[s->snid];
	if (ps->min < 0 || s->soff < ps->min) ps->min = s->soff;
	if (ps->max < 0 || s->soff + s->len > ps->max) ps->max = s->soff + s->len;
	if (ps->rank < 0) ps->rank = s->rank;
}

gfa_arc_t *add_arc1(gfa_t *g, uint32_t v, uint32_t w, int32_t ov, int32_t ow, int64_t link_id, int comp) // reference: gfa-base.c:148-168
{
	if (g->m_arc == g->n_arc) {
		uint64_t old_m = g->m_arc;
		g->m_arc = g->m_arc? g->m_arc << 1 : 16;
		g->arc = (gfa_arc_t*)realloc(g->arc, g->m_arc * sizeof(gfa_arc_t));
		memset(&g->arc[old_m], 0, (g->m_arc - old_m) * sizeof(gfa_arc_t));
		g->link_aux = (gfa_aux_t*)realloc(g->link_aux, g->m_arc * sizeof(gfa_aux_t));
		memset(&g->link_aux[old_m], 0, (g->m_arc - old_m) * sizeof(gfa_aux_t));
	}
	gfa_arc_t *a = &g->arc[g->n_arc++];
	a->v_lv = (uint64_t)v << 32;
	a->w = w, a->ov = ov, a->ow = ow, a->rank = -1;
	a->link_id = link_id >= 0? (uint64_t)link_id : g->n_arc - 1;
	if (link_id >= 0) a->rank = g->arc[link_id].rank;
	a->del = a->strong = 0;
	a->comp = comp;
	return a;
}

// tags of interest on one line: returns value text of TAG:T:... or 0
const char *find_tag(const std::vector<char*> &fld, size_t from, const char *tag, char type)
{
	for (size_t i = from; i < fld.size(); ++i) {
		const char *f = fld[i];
		if (strlen(f) >= 5 && f[0] == tag[0] && f[1] == tag[1] && f[2] == ':' && f[3] == type && f[4] == ':') return f + 5;
	}
	return 0;
}

void split_tab(char *s, std::vector<char*> &fld)
{
	fld.clear();
	char *p = s;
	for (;;) {
		fld.push_back(p);
		char *q = strchr(p, '\t');
		if (q == 0) break;
		*q = 0, p = q + 1;
	}
}

int parse_S(gfa_t *g, std::vector<char*> &fld) // reference: gfa-io.c:113-177
{
	if (fld.size() < 3) return -1;
	const char *seg = fld[1];
	char *seq = fld[2][0] == '*'? 0 : strdup(fld[2]);
	int32_t LN = -1;
	uint32_t len = 0;
	const char *t;
	if ((t = find_tag(fld, 3, "LN", 'i')) != 0) LN = atoi(t);
	if (seq == 0) { if (LN >= 0) len = (uint32_t)LN; }
	else len = (uint32_t)strlen(seq);
	int32_t sid = add_seg(g, seg);
	gfa_seg_t *s = &g->seg[sid];
	s->len = (int32_t)len, s->seq = seq;
	if (fld.size() > 3) {
		bool any = false;
		if ((t = find_tag(fld, 3, "SN", 'Z')) != 0) {
			s->snid = sseq_add(g, t), s->soff = 0;
			const char *so = find_tag(fld, 3, "SO", 'i');
			if (so) s->soff = atoi(so);
			any = true;
		}
		const char *sr = find_tag(fld, 3, "SR", 'i');
		if (sr) {
			s->rank = atoi(sr);
			if (s->rank > (int32_t)g->max_rank) g->max_rank = (uint32_t)s->rank;
			any = true;
		}
		// the reference calls gfa_sseq_update() whenever the line carries any tag at all
		(void)any;
		sseq_update(g, s);
	}
	return 0;
}

int parse_L(gfa_t *g, std::vector<char*> &fld) // reference: gfa-io.c:179-265
{
	if (fld.size() < 5) return -1;
	int oriv, oriw;
	int32_t ov = INT32_MAX, ow = INT32_MAX;
	if (fld[2][0] != '+' && fld[2][0] != '-') return -2;
	if (fld[4][0] != '+' && fld[4][0] != '-') return -2;
	oriv = fld[2][0] != '+', oriw = fld[4][0] != '+';
	size_t tag_from = 5;
	if (fld.size() >= 6) {
		char *q = fld[5];
		tag_from = 6;
		if (*q == '*') ov = ow = 0;
		else if (isdigit((unsigned char)*q)) {
			char *r;
			ov = (int32_t)strtol(q, &r, 10);
			if (isupper((unsigned char)*r)) {
				ov = ow = 0;
				do {
					long l = strtol(q, &q, 10);
					if (*q == 'M' || *q == 'D' || *q == 'N') ov += (int32_t)l;
					if (*q == 'M' || *q == 'I' || *q == 'S') ow += (int32_t)l;
					++q;
				} while (isdigit((unsigned char)*q));
			} else if (*r == ':') {
				ow = isdigit((unsigned char)*(r+1))? (int32_t)strtol(r+1, &r, 10) : INT32_MAX;
			} else return -1;
		} else if (*q == ':') {
			ov = INT32_MAX;
			ow = isdigit((unsigned char)*(q+1))? (int32_t)strtol(q+1, &q, 10) : INT32_MAX;
		} else return -1;
	} else ov = ow = 0;
	if (ov == INT32_MAX || ow == INT32_MAX) {
		fprintf(stderr, "[E::mgb200] L-lines with unknown overlap lengths are not supported\n");
		return -3;
	}
	uint32_t v = (uint32_t)add_seg(g, fld[1]) << 1 | (uint32_t)oriv;
	uint32_t w = (uint32_t)add_seg(g, fld[3]) << 1 | (uint32_t)oriw;
	gfa_arc_t *arc = add_arc1(g, v, w, ov, ow, -1, 0);
	const char *t;
	if ((t = find_tag(fld, tag_from, "SR", 'i')) != 0) arc->rank = atoi(t);
	if ((t = find_tag(fld, tag_from, "L1", 'i')) != 0) {
		int32_t l1 = atoi(t);
		g->seg[v>>1].len = g->seg[v>>1].len > ov + l1? g->seg[v>>1].len : ov + l1;
	}
	if ((t = find_tag(fld, tag_from, "L2", 'i')) != 0) {
		int32_t l2 = atoi(t);
		g->seg[w>>1].len = g->seg[w>>1].len > ow + l2? g->seg[w>>1].len : ow + l2;
	}
	return 0;
}

#define ARC_N(g, v) ((uint32_t)(g)->idx[(v)])
#define ARC_A(g, v) (&(g)->arc[(g)->idx[(v)] >> 32])

void fix_symm_add(gfa_t *g) // reference: gfa-base.c:267-303
{
	uint32_t v, n_vtx = g->n_seg * 2;
	uint64_t n_arc0 = g->n_arc;
	for (v = 0; v < n_vtx; ++v) {
		int nv = (int)ARC_N(g, v);
		gfa_arc_t *av = ARC_A(g, v);
		for (int i = 0; i < nv; ++i) {
			int j, nw;
			gfa_arc_t *aw, *avi = &av[i];
			if (avi->del || avi->comp) continue;
			nw = (int)ARC_N(g, avi->w ^ 1);
			aw = ARC_A(g, avi->w ^ 1);
			for (j = 0; j < nw; ++j) {
				gfa_arc_t *awj = &aw[j];
				if (awj->del || awj->comp) continue;
				if (awj->w == (v ^ 1) && awj->ov == avi->ow && awj->ow == avi->ov) {
					awj->comp = 1;
					awj->link_id = avi->link_id;
					break;
				}
			}
			if (j == nw) {
				gfa_arc_t *arc_old = g->arc, *arc_new;
				arc_new = add_arc1(g, avi->w ^ 1, v ^ 1, avi->ow, avi->ov, (int64_t)avi->link_id, 1);
				if (arc_old != g->arc) av = ARC_A(g, v);
				arc_new->rank = av[i].rank;
			}
		}
	}
	// NB: the reference re-sorts here only `if (n_vtx < gfa_n_vtx(g))`, which never holds (gfa-base.c:298-301): the
	// appended complement arcs stay unsorted until gfa_cleanup().  Mirrored on purpose -- one sort less changes tie order.
	(void)n_arc0;
}

void finalize(gfa_t *g) // reference: gfa-base.c:421-430
{
	for (uint32_t i = 0; i < g->n_seg; ++i) // gfa_fix_no_seg
		if (g->seg[i].len == 0) g->seg[i].del = 1;
	arc_sort(g);
	arc_index(g);
	// gfa_fix_semi_arc: nothing to do, unknown overlaps are rejected at parse time
	fix_symm_add(g);
	for (uint64_t k = 0; k < g->n_arc; ++k) { // gfa_fix_arc_len
		gfa_arc_t *a = &g->arc[k];
		uint32_t v = (uint32_t)(a->v_lv >> 32), w = a->w;
		const gfa_seg_t *sv = &g->seg[v>>1];
		if (!sv->del && sv->len < a->ov) a->ov = sv->len;
		if (sv->del || g->seg[w>>1].del) a->del = 1;
		else a->v_lv |= (uint64_t)(uint32_t)(sv->len - a->ov);
	}
	{ // gfa_cleanup = gfa_arc_rm + sort + index
		uint64_t e, n;
		for (e = n = 0; e < g->n_arc; ++e) {
			uint32_t u = (uint32_t)(g->arc[e].v_lv >> 32), v = g->arc[e].w;
			if (!g->arc[e].del && !g->seg[u>>1].del && !g->seg[v>>1].del) g->arc[n++] = g->arc[e];
		}
		if (n < g->n_arc) { free(g->idx); g->idx = 0; }
		g->n_arc = n;
		if (!arc_is_sorted(g)) {
			arc_sort(g);
			free(g->idx); g->idx = 0;
		}
		if (g->idx == 0) arc_index(g);
	}
}

} // namespace

extern "C" gfa_t *mgb_gfa_read(const char *fn)
{
	gzFile fp = gzopen(fn, "r");
	if (fp == 0) return 0;
	gfa_t *g = (gfa_t*)calloc(1, sizeof(gfa_t));
	g->h_names = new name_map_t();
	g->h_snames = new name_map_t();
	std::string line, fa_seq;
	std::vector<char> buf(1 << 16);
	std::vector<char*> fld;
	bool is_fa = false;
	int32_t fa_seg = -1;
	auto finish_fa = [&]() {
		if (fa_seg < 0) return;
		gfa_seg_t *s = &g->seg[fa_seg];
		s->seq = strdup(fa_seq.c_str());
		s->len = (int32_t)fa_seq.size();
		sseq_update(g, s);
	};
	bool eof = false;
	while (!eof) {
		line.clear();
		for (;;) { // read one line of any length
			if (gzgets(fp, buf.data(), (int)buf.size()) == 0) { eof = true; break; }
			size_t l = strlen(buf.data());
			line.append(buf.data(), l);
			if (l > 0 && buf[l-1] == '\n') break;
		}
		if (eof && line.empty()) break;
		while (!line.empty() && (line.back() == '\n' || line.back() == '\r')) line.pop_back();
		if (!line.empty() && line[0] == '>') { // FASTA header (reference: gfa-io.c:267-281)
			is_fa = true;
			finish_fa();
			size_t e = 1;
			while (e < line.size() && !isspace((unsigned char)line[e])) ++e;
			std::string nm = line.substr(1, e - 1);
			char sbuf[32];
			snprintf(sbuf, sizeof(sbuf), "s%d", (int)g->n_seg + 1);
			fa_seg = add_seg(g, sbuf);
			gfa_seg_t *seg = &g->seg[fa_seg];
			seg->snid = sseq_add(g, nm.c_str());
			seg->soff = seg->rank = 0;
			fa_seq.clear();
			continue;
		} else if (is_fa) {
			if (line.size() >= 3 && line[1] == '\t') { finish_fa(); fa_seg = -1; is_fa = false; }
			else { fa_seq += line; continue; }
		}
		if (line.size() < 3 || line[1] != '\t') continue;
		if (line[0] == 'S' || line[0] == 'L') {
			std::vector<char> tmp(line.begin(), line.end());
			tmp.push_back(0);
			split_tab(tmp.data(), fld);
			int ret = line[0] == 'S'? parse_S(g, fld) : parse_L(g, fld);
			if (ret < 0) fprintf(stderr, "[E::mgb200] invalid %c-line (error code %d)\n", line[0], ret);
		}
	}
	if (is_fa) finish_fa();
	gzclose(fp);
	finalize(g);
	return g;
}

extern "C" void mgb_gfa_destroy(gfa_t *g)
{
	if (g == 0) return;
	delete (name_map_t*)g->h_names;
	delete (name_map_t*)g->h_snames;
	for (uint32_t i = 0; i < g->n_seg; ++i) { free(g->seg[i].name); free(g->seg[i].seq); }
	for (uint32_t i = 0; i < g->n_sseq; ++i) free(g->sseq[i].name);
	free(g->idx); free(g->seg); free(g->arc); free(g->link_aux); free(g->sseq);
	free(g);
}

// ---------------------------------------------------------------------------------------------------------------
// GAF writer
// ---------------------------------------------------------------------------------------------------------------

namespace {

struct Str { char *b; size_t l, m; }; // local copy of the caller's buffer: keeps pointer and length in registers

inline void s_reserve(Str &s, size_t extra)
{
	if (s.l + extra + 1 > s.m) {
		size_t c = s.m? s.m : 256;
		while (c < s.l + extra + 1) c <<= 1;
		s.b = (char*)realloc(s.b, c);
		s.m = c;
	}
}
inline void s_putc(Str &s, char c) { s_reserve(s, 1); s.b[s.l++] = c; }
inline void s_puts(Str &s, const char *p) { size_t l = strlen(p); s_reserve(s, l); memcpy(s.b + s.l, p, l); s.l += l; }
inline void s_putn(Str &s, const char *p, size_t l) { s_reserve(s, l); memcpy(s.b + s.l, p, l); s.l += l; }
inline void s_putd(Str &s, int c)
{
	char b[16];
	int l = 0;
	unsigned x = c >= 0? (unsigned)c : (unsigned)(-c);
	do { b[l++] = (char)(x % 10 + '0'); x /= 10; } while (x > 0);
	if (c < 0) b[l++] = '-';
	s_reserve(s, (size_t)l);
	for (int i = l - 1; i >= 0; --i) s.b[s.l++] = b[i];
}
// unchecked variants for the bulk fields (capacity reserved by the caller)
inline void u_putd(Str &s, unsigned x)
{
	char b[12];
	int l = 0;
	do { b[l++] = (char)(x % 10 + '0'); x /= 10; } while (x > 0);
	while (l > 0) s.b[s.l++] = b[--l];
}
inline void s_seg(Str &s, char sign, const char *name, int st, int en) { s_putc(s, sign); s_puts(s, name); s_putc(s, ':'); s_putd(s, st); s_putc(s, '-'); s_putd(s, en); }

unsigned char g_comp[256];
bool g_comp_init = false;
void init_comp()
{
	static const char *from = "ABCDEFGHIJKLMNOPQRSTUVWXYZ", *to = "TVGHEFCDIJMLKNOPQYSAABWXRZ";
	for (int i = 0; i < 256; ++i) g_comp[i] = (unsigned char)i;
	for (int i = 0; i < 26; ++i) {
		g_comp[(unsigned char)from[i]] = (unsigned char)to[i];
		g_comp[(unsigned char)(from[i] + 32)] = (unsigned char)(to[i] + 32);
	}
	g_comp_init = true;
}

const uint64_t F_FRAG_MERGE = 0x80, F_VERTEX_COOR = 0x800, F_PRINT_2ND = 0x2000, F_SHOW_UNMAP = 0x100000, F_NO_COMP_PATH = 0x200000;
const uint64_t F_WRITE_LCHAIN = 0x800000, F_WRITE_MZ = 0x1000000;

} // namespace

namespace mgb {
// The `dv:f` field of a record as format.c:200-205 prints it: absent unless 0 <= div <= 1, "0" for 0, else "%.4f".  Writes the
// field with its leading tab to b (16 bytes are enough) and returns its length, 0 when absent.  mgb_write_gaf() and the text route
// of the engine (mgb_map_batch_gaf) both print it from here.
int gaf_dv_text(float div, char *b)
{
	if (!(div >= 0.0f && div <= 1.0f)) return 0;
	memcpy(b, "\tdv:f:", 6);
	if (div == 0.0f) { b[6] = '0'; return 7; }
	return 6 + snprintf(b + 6, 10, "%.4f", div);
}
}

extern "C" void mgb_write_gaf(char **buf, size_t *len, size_t *cap, const gfa_t *g, const mg_gchains_t *gs, int32_t qlen, const char *qname, uint64_t flag)
{
	Str s = { *buf, *len, *cap };
	struct Sync { Str &s; char **b; size_t *l, *m; ~Sync() { *b = s.b, *l = s.l, *m = s.m; } } sync_back = { s, buf, len, cap };
	int32_t rev_sign = 0; // sticky across the records of one read, like the reference (format.c:123)
	if (!g_comp_init) init_comp();
	if ((gs == 0 || gs->n_gc == 0) && (flag & F_SHOW_UNMAP)) {
		s_puts(s, qname); s_putc(s, '\t'); s_putd(s, qlen); s_puts(s, "\t0\t0\t*\t*\t0\t0\t0\t0\t0\t0\n");
		s.b[s.l] = 0;
		return;
	}
	if (gs == 0) return;
	for (int32_t i = 0; i < gs->n_gc; ++i) {
		const mg_gchain_t *p = &gs->gc[i];
		size_t sign_pos;
		int32_t compact;
		if (p->id != p->parent && !(flag & F_PRINT_2ND)) continue;
		if (p->cnt == 0) continue;
		s_puts(s, qname);
		s_putc(s, '\t'); s_putd(s, qlen); s_putc(s, '\t'); s_putd(s, p->qs); s_putc(s, '\t'); s_putd(s, p->qe); s_puts(s, "\t+\t");
		sign_pos = s.l - 2;
		if (flag & F_VERTEX_COOR) {
			compact = 0;
			for (int32_t j = 0; j < p->cnt; ++j) {
				const mg_llchain_t *q = &gs->lc[p->off + j];
				s_putc(s, "><"[q->v & 1]); s_puts(s, g->seg[q->v >> 1].name);
			}
		} else {
			int32_t last_pnid = -1, st = -1, en = -1, rev = -1;
			compact = flag & F_NO_COMP_PATH? 0 : 1;
			for (int32_t j = 0; j < p->cnt; ++j) {
				const mg_llchain_t *q = &gs->lc[p->off + j];
				const gfa_seg_t *t = &g->seg[q->v >> 1];
				if (t->snid < 0) {
					compact = 0;
					if (last_pnid >= 0) s_seg(s, "><"[rev], g->sseq[last_pnid].name, st, en);
					last_pnid = -1, st = -1, en = -1, rev = -1;
					s_putc(s, "><"[q->v & 1]); s_puts(s, g->seg[q->v >> 1].name);
				} else {
					int cont = 0;
					if (last_pnid >= 0 && t->snid == last_pnid && (int32_t)(q->v & 1) == rev) {
						if (!(q->v & 1)) {
							if (t->soff == en) en = t->soff + t->len, cont = 1;
						} else {
							if (t->soff + t->len == st) st = t->soff, cont = 1;
						}
					}
					if (cont == 0) {
						if (last_pnid >= 0) compact = 0;
						if (last_pnid >= 0) s_seg(s, "><"[rev], g->sseq[last_pnid].name, st, en);
						last_pnid = t->snid, rev = (int32_t)(q->v & 1), st = t->soff, en = st + t->len;
					}
				}
			}
			if (last_pnid >= 0) {
				if (g->sseq[last_pnid].rank != 0 || g->sseq[last_pnid].min != 0) compact = 0;
				if (!compact) s_seg(s, "><"[rev], g->sseq[last_pnid].name, st, en);
			} else compact = 0;
		}
		if (compact) {
			int32_t rev = (int32_t)(gs->lc[p->off].v & 1);
			const gfa_seg_t *t = &g->seg[gs->lc[rev? p->off + p->cnt - 1 : p->off].v >> 1];
			const gfa_sseq_t *ps = &g->sseq[t->snid];
			s_puts(s, ps->name); s_putc(s, '\t'); s_putd(s, ps->max); s_putc(s, '\t');
			if (rev) {
				rev_sign = 1;
				s.b[sign_pos] = '-';
				s_putd(s, t->soff + (p->plen - p->pe)); s_putc(s, '\t'); s_putd(s, t->soff + (p->plen - p->ps));
			} else {
				s_putd(s, t->soff + p->ps); s_putc(s, '\t'); s_putd(s, t->soff + p->pe);
			}
		} else { s_putc(s, '\t'); s_putd(s, p->plen); s_putc(s, '\t'); s_putd(s, p->ps); s_putc(s, '\t'); s_putd(s, p->pe); }
		if (p->p) { s_putc(s, '\t'); s_putd(s, p->p->mlen); s_putc(s, '\t'); s_putd(s, p->p->blen); s_putc(s, '\t'); s_putd(s, (int)p->mapq); }
		else { s_putc(s, '\t'); s_putd(s, p->mlen); s_putc(s, '\t'); s_putd(s, p->blen); s_putc(s, '\t'); s_putd(s, (int)p->mapq); }
		s_puts(s, "\ttp:A:"); s_putc(s, p->id == p->parent? 'P' : 'S');
		if (p->p) { s_puts(s, "\tNM:i:"); s_putd(s, p->p->blen - p->p->mlen); }
		s_puts(s, "\tcm:i:"); s_putd(s, p->n_anchor); s_puts(s, "\ts1:i:"); s_putd(s, p->score); s_puts(s, "\ts2:i:"); s_putd(s, p->subsc);
		{
			char b[16];
			s_putn(s, b, (size_t)mgb::gaf_dv_text(p->div, b));
		}
		if (p->p) {
			s_puts(s, "\tcg:Z:");
			s_reserve(s, (size_t)p->p->n_cigar * 12 + 16);
			if (rev_sign)
				for (int32_t j = p->p->n_cigar - 1; j >= 0; --j) { u_putd(s, (unsigned)(p->p->cigar[j] >> 4)); s.b[s.l++] = "MIDNSHP=XB"[p->p->cigar[j] & 0xf]; }
			else
				for (int32_t j = 0; j < p->p->n_cigar; ++j) { u_putd(s, (unsigned)(p->p->cigar[j] >> 4)); s.b[s.l++] = "MIDNSHP=XB"[p->p->cigar[j] & 0xf]; }
		}
		if (p->ds.ds) {
			s_puts(s, "\tds:Z:");
			s_reserve(s, (size_t)p->ds.len + 16);
			if (rev_sign) {
				const char *ds = p->ds.ds;
				for (int32_t k = p->ds.n_off - 1; k >= 0; --k) {
					int32_t off = p->ds.off[k], en;
					s_putc(s, ds[off]);
					en = k < p->ds.n_off - 1? p->ds.off[k+1] : p->ds.len;
					if (ds[off] == ':') {
						s_putn(s, ds + off + 1, (size_t)(en - off - 1));
					} else if (ds[off] == '*') {
						for (int32_t j = off + 1; j < en; ++j) s_putc(s, (char)g_comp[(uint8_t)ds[j]]);
					} else {
						for (int32_t j = en - 1; j >= off + 1; --j) {
							if (ds[j] == '[') s_putc(s, ']');
							else if (ds[j] == ']') s_putc(s, '[');
							else s_putc(s, (char)g_comp[(uint8_t)ds[j]]);
						}
					}
				}
			} else s_putn(s, p->ds.ds, (size_t)p->ds.len);
		}
		s_putc(s, '\n');
		if (flag & F_WRITE_LCHAIN) { // -S / --write-mz (format.c:252-289)
			char b[16];
			for (int32_t j = 0; j < p->cnt; ++j) {
				const mg_llchain_t *lc = &gs->lc[p->off + j];
				s_puts(s, "*\t"); s_putc(s, "><"[lc->v & 1]); s_puts(s, g->seg[lc->v >> 1].name); s_putc(s, '\t'); s_putd(s, g->seg[lc->v >> 1].len); s_putc(s, '\t'); s_putd(s, lc->cnt);
				if (lc->cnt > 0) {
					double div;
					int32_t q_span = (int32_t)(gs->a[lc->off].y >> 32 & 0xff);
					int32_t n = (int32_t)(gs->a[lc->off + lc->cnt - 1].x >> 32) - (int32_t)(gs->a[lc->off].x >> 32) + 1;
					div = n == lc->cnt? 0.0 : (n > lc->cnt? log((double)n / lc->cnt) : log((double)lc->cnt / n)) / q_span;
					if (div == 0.0) b[0] = '0', b[1] = 0;
					else snprintf(b, 16, "%.4f", div);
					s_putc(s, '\t'); s_puts(s, b);
					s_putc(s, '\t'); s_putd(s, (int32_t)gs->a[lc->off].x + 1 - q_span); s_putc(s, '\t'); s_putd(s, (int32_t)gs->a[lc->off + lc->cnt - 1].x + 1);
					s_putc(s, '\t'); s_putd(s, (int32_t)gs->a[lc->off].y + 1 - q_span); s_putc(s, '\t'); s_putd(s, (int32_t)gs->a[lc->off + lc->cnt - 1].y + 1);
					if (flag & F_WRITE_MZ) {
						int32_t last = (int32_t)gs->a[lc->off].x + 1 - q_span;
						s_putc(s, '\t'); s_putd(s, q_span); s_putc(s, '\t');
						for (int32_t k = 1; k < lc->cnt; ++k) {
							int32_t x = (int32_t)gs->a[lc->off + k].x + 1 - q_span;
							if (k > 1) s_putc(s, ',');
							s_putd(s, x - last);
							last = x;
						}
						last = (int32_t)gs->a[lc->off].y + 1 - q_span;
						s_putc(s, '\t');
						for (int32_t k = 1; k < lc->cnt; ++k) {
							int32_t x = (int32_t)gs->a[lc->off + k].y + 1 - q_span;
							if (k > 1) s_putc(s, ',');
							s_putd(s, x - last);
							last = x;
						}
					}
				}
				s_putc(s, '\n');
			}
		}
	}
	s_reserve(s, 1);
	s.b[s.l] = 0;
	(void)F_FRAG_MERGE;
}

// GAF text for a whole batch, input order preserved (the reference writes from one thread, gmap.c:101-141; here the
// records are formatted by several host threads into per-thread buffers, which the same threads then copy to their
// place in the output).  The per-thread buffers are kept between calls, and a caller that hands back the previous
// output buffer (*out with its *out_cap) gets it reused: in steady state no page is touched for the
// first time, which is what the formatting of ~100 MB of text otherwise mostly waits for.
#include <thread>
#include <mutex>
#include <functional>
#include "mgb_hostpool.h"
extern "C" void mgb_write_gaf_batch(const gfa_t *g, int n_reads, mg_gchains_t *const *gcs, const int *qlens, const char *const *names,
									uint64_t flag, int n_threads, char **out, size_t *out_len, size_t *out_cap)
{
	struct Part { char *buf; size_t len, cap; };
	static std::mutex mtx;
	static std::vector<Part> pool;
	std::lock_guard<std::mutex> lock(mtx);
	if (n_threads <= 0) { n_threads = (int)std::thread::hardware_concurrency(); if (n_threads > 16) n_threads = 16; if (n_threads < 1) n_threads = 1; }
	if (n_reads < 256) n_threads = 1;
	if ((int)pool.size() < n_threads) pool.resize((size_t)n_threads, Part{0, 0, 0});
	const int64_t chunk = ((int64_t)n_reads + n_threads - 1) / n_threads;
	static mgb::HostPool workers; // the writer's own workers (the engine may be mapping the next batch on its pool meanwhile)
	auto run = [&](const std::function<void(int)> &fn) {
		if (n_threads == 1) { fn(0); return; }
		workers.run(n_threads, n_threads, [&](int64_t t) { fn((int)t); });
	};
	run([&](int t) {
		int64_t b = t * chunk, e = b + chunk < n_reads? b + chunk : n_reads;
		Part &p = pool[(size_t)t];
		p.len = 0;
		for (int64_t i = b; i < e; ++i)
			mgb_write_gaf(&p.buf, &p.len, &p.cap, g, gcs[i], qlens[i], names && names[i]? names[i] : "*", flag);
	});
	size_t tot = 0;
	std::vector<size_t> at((size_t)n_threads, 0);
	for (int t = 0; t < n_threads; ++t) at[(size_t)t] = tot, tot += pool[(size_t)t].len;
	char *o = out_cap? *out : 0;
	size_t cap = o? *out_cap : 0;
	if (cap < tot + 1) {
		free(o);
		cap = tot + tot / 8 + 1;
		o = (char*)malloc(cap);
	}
	run([&](int t) { const Part &p = pool[(size_t)t]; if (p.len) memcpy(o + at[(size_t)t], p.buf, p.len); });
	o[tot] = 0;
	*out = o, *out_len = tot;
	if (out_cap) *out_cap = cap;
}

// ---------------------------------------------------------------------------------------------------------------
// input side: a whole FASTA/FASTQ file (plain or gzip) as the arrays mg_map_batch() takes
// (reference: bseq.c:46-98 mg_bseq_read + the upper-casing of gmap.c:77-84; kseq.h's rules: the name ends at the first
// white space, sequence lines are joined, a FASTQ record's quality is skipped by length)
// ---------------------------------------------------------------------------------------------------------------
extern "C" mgb_reads_t *mgb_reads_load(const char *fn, int64_t max_bases)
{
	gzFile fp = fn && strcmp(fn, "-")? gzopen(fn, "rb") : gzdopen(0, "rb");
	if (fp == 0) return 0;
	std::vector<char> raw;
	{
		char buf[1 << 16];
		int n;
		gzbuffer(fp, 1 << 20);
		while ((n = gzread(fp, buf, sizeof(buf))) > 0) raw.insert(raw.end(), buf, buf + n);
		gzclose(fp);
	}
	mgb_reads_t *r = (mgb_reads_t*)calloc(1, sizeof(mgb_reads_t));
	// the records are compacted in place: name\0seq\0 follow each other in one block that the arrays point into
	r->block = (char*)malloc(raw.size() + 2);
	std::vector<size_t> name_off, seq_off;
	std::vector<int> len;
	size_t w = 0, i = 0;
	const size_t n = raw.size();
	int64_t bases = 0;
	while (i < n && raw[i] != '>' && raw[i] != '@') ++i; // kseq skips to the first header
	while (i < n && (max_bases <= 0 || bases < max_bases)) {
		const char head = raw[i++];
		name_off.push_back(w);
		while (i < n && !isspace((unsigned char)raw[i])) r->block[w++] = raw[i++];
		r->block[w++] = 0;
		while (i < n && raw[i] != '\n') ++i; // comment
		seq_off.push_back(w);
		size_t l = 0;
		while (i < n) { // sequence lines up to the next header ('+' ends a FASTQ sequence)
			if (raw[i] == '\n' || raw[i] == '\r') { ++i; continue; }
			if (raw[i - 1] == '\n' && (raw[i] == '>' || raw[i] == '+' || raw[i] == '@')) break;
			const unsigned char c = (unsigned char)raw[i++];
			r->block[w++] = (char)(c >= 'a' && c <= 'z'? c - 32 : c), ++l; // gmap.c:81
		}
		r->block[w++] = 0;
		len.push_back((int)l), bases += (int64_t)l;
		if (head == '@' && i < n && raw[i] == '+') { // quality: as many characters as bases
			while (i < n && raw[i] != '\n') ++i;
			size_t q = 0;
			while (i < n && q < l) { if (raw[i] != '\n' && raw[i] != '\r') ++q; ++i; }
			while (i < n && raw[i] != '\n') ++i;
		}
		while (i < n && raw[i] != '>' && raw[i] != '@') ++i;
	}
	r->n_reads = (int64_t)len.size(), r->n_bases = bases;
	r->name = (const char**)malloc(sizeof(char*) * (len.size() + 1)), r->seq = (const char**)malloc(sizeof(char*) * (len.size() + 1)), r->len = (int*)malloc(sizeof(int) * (len.size() + 1));
	for (size_t k = 0; k < len.size(); ++k) r->name[k] = r->block + name_off[k], r->seq[k] = r->block + seq_off[k], r->len[k] = len[k];
	return r;
}

extern "C" void mgb_reads_free(mgb_reads_t *r)
{
	if (r == 0) return;
	free(r->block); free((void*)r->name); free((void*)r->seq); free(r->len); free(r);
}
