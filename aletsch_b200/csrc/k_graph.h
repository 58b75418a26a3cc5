// Stage 2 kernel: one CTA per bundle builds the splice graph from the bundle's evidence
// (chain sets hcst + fcst, coverage segments, bounds, strand).
//
// Reference semantics reproduced (rnacore/graph_builder.cc):
//   build_junctions            :46-125   chains exploded in chain-set order, AI3 counts summed per (l, r),
//                                        junction order = chain_set insertion order of the temporary jcst
//   remove_opposite_junctions  :128-175  provably a no-op (junction::nm is always 0, rnacore/junction.cc:26:
//                                        both ratios are 0.0 and the strict '<' never holds)
//   build_regions              :177-224  boundary map, LEFT_RIGHT_SPLICE resolution
//   region::region             rnacore/region.cc:22-169 (join map, smoothing, empty_subregion, pexons, stubs)
//   evaluate_rectangle         rnacore/interval_map.cc:166-195 (int32 sum, double ave / dev in segment order)
//   build_partial_exons / classify / link   :226-297, :477-514
//   build_splice_graph         :299-426  (vertex weights, junction / boundary / adjacency edges, insertion order)
//   refine_splice_graph        rnacore/graph_reviser.cc:899-914
#ifndef ALETSCH_B200_CSRC_K_GRAPH_H
#define ALETSCH_B200_CSRC_K_GRAPH_H

#include "dev.h"
#include "blockops.h"

namespace agpu {

// boundary types, util/constants.h:21-28
#define START_BOUNDARY 1
#define END_BOUNDARY 2
#define LEFT_SPLICE 3
#define RIGHT_SPLICE 4
#define LEFT_RIGHT_SPLICE 5

struct chains_view
{
	int present;
	const int64_t *elem_off;     // [NB+1] scratch base of the bundle's chain records
	const int32_t *n_chains;     // [NB]
	const int32_t *c_rep;        // chain record -> representative element (bundle-local)
	const int32_t *c_cnt;        // [3 per chain record]
	const int32_t *elem_len;     // per element: number of coordinates
	const u32 *voff32;           // per element: offset of its coordinates in val (one of the two)
	const int64_t *voff64;
	const int32_t *val;
	DEV int count(int b) const { return present ? n_chains[b] : 0; }
	DEV int len(int b, int k) const { return elem_len[elem_off[b] + c_rep[elem_off[b] + k]]; }
	DEV const int32_t *ptr(int b, int k) const
	{
		int64_t e = elem_off[b] + c_rep[elem_off[b] + k];
		return val + (voff64 ? voff64[e] : (int64_t)voff32[e]);
	}
	DEV const int32_t *cnt(int b, int k) const { return c_cnt + (elem_off[b] + k) * 3; }
};

struct graph_in
{
	int32_t n;
	const int32_t *lpos, *rpos;
	const uint8_t *strand;
	chains_view hc, fc;
	const int64_t *seg_off;
	const int32_t *seg_l, *seg_r, *seg_c;
	const int64_t *seg_nhead, *seg_psum;   // batch-wide side tables (coverage_scan): next run-opening segment, prefix sums of len * cov
};

struct graph_dev
{
	// upper-bound layout: bundle b owns [off[b], off[b+1]) of each family
	const int64_t *junc_off, *pex_off, *edge_off, *iarena_off, *karena_off;
	int32_t *iarena;
	u64 *karena;
	int32_t *n_junc, *n_pex, *n_edge;
	int32_t *j_l, *j_r, *j_cnt, *j_xs0, *j_xs1, *j_xs2, *j_strand, *j_lexon, *j_rexon;
	int32_t *p_l, *p_r, *p_lt, *p_rt, *p_regional, *p_type;
	double *p_ave, *p_dev, *p_max;
	// vertices of bundle b live at pex_off[b] + 2 * b ... (P + 2 of them)
	int32_t *v_l, *v_r, *v_len, *v_type, *v_regional, *v_brk;   // v_brk: prefix count of non-continuous steps
	double *v_w, *v_dev, *v_max;
	int32_t *e_s, *e_t, *e_strand;
	double *e_w;
	// alive edges sorted by (target, source): in_off has V + 1 entries per bundle at pex_off[b] + 3 * b
	int32_t *in_off, *in_src, *in_eid;
	// alive edges sorted by (source, target): out_off likewise
	int32_t *out_off, *out_dst, *out_eid;
	// bundle -> graph index when the graphs belong to another batch (assembler::bridge: every member bundle of a cluster works
	// against the graph of the combined bundle, meta/assembler.cc:989-998); NULL: graph b belongs to bundle b; < 0: no graph
	const int32_t *remap;
	int *err;
};

HD int graph_index(const graph_dev &g, int b) { return g.remap ? g.remap[b] : b; }
HD int64_t vert_base(const graph_dev &g, int b) { return g.pex_off[b] + 2 * (int64_t)b; }
HD int64_t voff_base(const graph_dev &g, int b) { return g.pex_off[b] + 3 * (int64_t)b; }

// per bundle upper bounds for the scratch / output layout
KERNEL k_graph_bounds(graph_in in, int64_t *ub_junc, int64_t *ub_pex, int64_t *ub_edge, int64_t *ub_iarena, int64_t *ub_karena)
{
	SHARED int s_inst;
	for(int b = blockIdx.x; b < in.n; b += gridDim.x)
	{
		if(threadIdx.x == 0) s_inst = 0;
		BLOCK_SYNC();
		int nh = in.hc.count(b), nf = in.fc.count(b);
		int acc = 0;
		for(int k = threadIdx.x; k < nh + nf; k += blockDim.x)
		{
			int len = k < nh ? in.hc.len(b, k) : in.fc.len(b, k - nh);
			if(len > 0 && (len & 1) == 0) acc += len / 2;
		}
		atomicAdd(&s_inst, acc);
		BLOCK_SYNC();
		if(threadIdx.x == 0)
		{
			int64_t ninst = s_inst;
			int64_t S = in.seg_off[b + 1] - in.seg_off[b];
			int64_t J = ninst, NB = 2 * J + 2, NR = NB, P = S + 2 * NR + 2;
			ub_junc[b] = J;
			ub_pex[b] = P;
			ub_edge[b] = J + 3 * P + 2;
			ub_iarena[b] = (nh + nf) + 20 * ninst + 10 * P + 128;
			ub_karena[b] = 6 * ninst + (J + 3 * P + 2) + 64;
		}
		BLOCK_SYNC();
	}
}

struct seg_view
{
	const int32_t *l, *r, *c;
	int n;
	const int64_t *nhead;      // nhead[i] - base = first index > i whose segment does not touch its predecessor (<= n)
	const int64_t *psum;       // psum[i] = sum over the batch's segments before i of the int32 products (r - l) * c
	int64_t base;              // index of the bundle's first segment in the batch-wide tables
};

// locate_boundary_iterators (rnacore/interval_map.cc:70-87): index range of the segments lying fully inside [x, y)
DEV bool segs_inside(const seg_view &s, int32_t x, int32_t y, int &i0, int &i1)
{
	i0 = lower_bound_idx(s.l, s.n, x);                 // first segment with lower >= x
	if(i0 >= s.n || s.r[i0] > y) return false;
	i1 = upper_bound_idx(s.r, s.n, y) - 1;             // last segment with upper <= y
	if(i1 < 0 || s.l[i1] < x) return false;
	return i0 <= i1;
}

// compute_sum_overlap (rnacore/interval_map.cc:128-149) over the segments a..e: int32 arithmetic
DEV int32_t seg_sum(const seg_view &s, int a, int e) { return (int32_t)(u32)(unsigned long long)(s.psum[e + 1] - s.psum[a]); }

// evaluate_rectangle (rnacore/interval_map.cc:166-195) over [ll, rr) whose inside segments are a..e (none if e < a)
DEV void evaluate_rectangle(const seg_view &s, int32_t ll, int32_t rr, int a, int e, double &ave, double &dev, double &mx)
{
	ave = 0; dev = 1; mx = 0;
	if(e < a) return;
	int32_t sum = seg_sum(s, a, e);
	ave = 1.0 * sum / (rr - ll);
	int32_t m = 0;
	double var = 0;
	// the reference's accumulation order; four independent terms are formed at a time, then added in order
	int i = a;
	for(; i + 3 <= e; i += 4)
	{
		int32_t c0 = s.c[i], c1 = s.c[i + 1], c2 = s.c[i + 2], c3 = s.c[i + 3];
		int32_t n0 = s.r[i] - s.l[i], n1 = s.r[i + 1] - s.l[i + 1], n2 = s.r[i + 2] - s.l[i + 2], n3 = s.r[i + 3] - s.l[i + 3];
		double d0 = c0 - ave, d1 = c1 - ave, d2 = c2 - ave, d3 = c3 - ave;
		double t0 = d0 * d0 * n0, t1 = d1 * d1 * n1, t2 = d2 * d2 * n2, t3 = d3 * d3 * n3;
		int32_t m01 = c0 > c1 ? c0 : c1, m23 = c2 > c3 ? c2 : c3;
		int32_t m4 = m01 > m23 ? m01 : m23;
		if(m4 > m) m = m4;
		var += t0; var += t1; var += t2; var += t3;
	}
	for(; i <= e; i++)
	{
		int32_t c = s.c[i];
		if(c > m) m = c;
		double d = c - ave;
		var += d * d * (s.r[i] - s.l[i]);
	}
	mx = 1.0 * m;
	dev = sqrt(var / (rr - ll));
}

// region::empty_subregion (rnacore/region.cc:88-107) for the run [p1, p2) made of the segments a..e
DEV bool empty_subregion(const seg_view &s, int32_t p1, int32_t p2, int a, int e, int min_len, double min_overlap)
{
	if(p2 - p1 < min_len) return true;
	if(e < a) return true;
	int32_t sum = seg_sum(s, a, e);
	double ratio = sum * 1.0 / (p2 - p1);
	if(ratio < min_overlap) return true;
	return false;
}

struct pexon_sink
{
	int emit;                  // 0: count only
	int n;
	int32_t *l, *r, *lt, *rt;
	double *ave, *dev, *mx;
	DEV void push(int32_t pl, int32_t pr, int plt, int prt, double a, double d, double m)
	{
		if(emit) { l[n] = pl; r[n] = pr; lt[n] = plt; rt[n] = prt; ave[n] = a; dev[n] = d; mx[n] = m; }
		n++;
	}
};

// iterates the runs of region::jmap after build_join_interval_map (+ smooth_join_interval_map); every run comes with the
// index range a..e of the segments inside it
struct run_iter
{
	const seg_view &s;
	int i, i1;
	bool any, smooth;
	int32_t lpos, rpos, gap;
	// pending raw run
	bool have_raw;
	int32_t raw_l, raw_r;
	int raw_a, raw_e;
	bool tail_done;
	int32_t prev_end;          // `p` of smooth_join_interval_map

	DEV run_iter(const seg_view &sv, int32_t lp, int32_t rp, bool sm, int32_t g) : s(sv), smooth(sm), lpos(lp), rpos(rp), gap(g)
	{
		int a = 0, b = -1;
		any = segs_inside(s, lp, rp, a, b);
		i = a; i1 = b;
		have_raw = false;
		tail_done = false;
		prev_end = lp;
	}

	DEV bool next_raw(int32_t &l, int32_t &r, int &a, int &e)
	{
		if(!any || i > i1) return false;
		a = i;
		e = (int)(s.nhead[i] - s.base) - 1;                // touching segments join (all values are 1)
		if(e > i1) e = i1;
		l = s.l[a]; r = s.r[e];
		i = e + 1;
		return true;
	}

	// next run of the (smoothed) join map
	DEV bool next(int32_t &l, int32_t &r, int &a, int &e)
	{
		if(!smooth) return next_raw(l, r, a, e);
		// smoothing (rnacore/region.cc:60-86): the stretch between the previous run (or lpos) and a run is filled
		// when it is at most min_subregion_gap long; likewise the stretch between the last run and rpos
		int32_t cl, cr;
		if(have_raw) { cl = raw_l; cr = raw_r; a = raw_a; e = raw_e; have_raw = false; }
		else if(!next_raw(cl, cr, a, e))
		{
			if(tail_done) return false;
			tail_done = true;
			// no run is pending: the tail stretch [prev_end, rpos) becomes a run of its own only if nothing precedes it
			// (otherwise it was merged below); this happens when the region holds no run at all
			if(prev_end == lpos && prev_end < rpos && rpos - prev_end <= gap) { l = prev_end; r = rpos; a = 0; e = -1; prev_end = rpos; return true; }
			return false;
		}
		if(cl - prev_end <= gap) cl = prev_end;              // fill [p, p1); at the region start this extends to lpos
		// absorb following runs whose gap to the current end is small
		while(true)
		{
			int32_t nl, nr;
			int na, ne;
			if(!next_raw(nl, nr, na, ne))
			{
				tail_done = true;
				if(cr < rpos && rpos - cr <= gap) cr = rpos;
				break;
			}
			if(nl - cr <= gap) { cr = nr; e = ne; continue; }
			raw_l = nl; raw_r = nr; raw_a = na; raw_e = ne; have_raw = true;
			break;
		}
		prev_end = cr;
		l = cl; r = cr;
		return true;
	}
};

// region::region + build_partial_exons (rnacore/region.cc:22-29, :109-169)
DEV void region_pexons(const seg_view &s, int32_t lpos, int32_t rpos, int ltype, int rtype,
		int min_gap, int min_len, double min_overlap, double min_weight, pexon_sink &out)
{
	bool smooth = (ltype == RIGHT_SPLICE && rtype == LEFT_SPLICE);
	run_iter it(s, lpos, rpos, smooth, min_gap);
	// the first run: is the join map empty / does the run span the whole region?
	int32_t p1 = 0, p2 = 0;
	int a = 0, e = -1;
	bool nonempty = it.next(p1, p2, a, e);
	if(!nonempty && rpos == lpos + 1 && (ltype == END_BOUNDARY || rtype == START_BOUNDARY))
	{
		out.push(lpos, rpos, ltype, rtype, min_weight, 1.0, -1.0);
		return;
	}
	if(nonempty && p1 == lpos && p2 == rpos)
	{
		double av = 0, d = 1, m = 0;
		if(out.emit) evaluate_rectangle(s, lpos, rpos, a, e, av, d, m);
		out.push(lpos, rpos, ltype, rtype, av, d, m);
		return;
	}
	// jmap.find(ROI(lpos, lpos + 1)) == end  <=>  no run starts at lpos (runs lie inside [lpos, rpos))
	if(ltype == RIGHT_SPLICE && !(nonempty && p1 == lpos))
		out.push(lpos, lpos + 1, ltype, END_BOUNDARY, min_weight, 1.0, -1.0);
	bool covers_end = false;
	for(bool have = nonempty; have; have = it.next(p1, p2, a, e))
	{
		if(p2 == rpos) covers_end = true;
		bool b = empty_subregion(s, p1, p2, a, e, min_len, min_overlap);
		if(p1 == lpos && ltype == RIGHT_SPLICE) b = false;
		if(p2 == rpos && rtype == LEFT_SPLICE) b = false;
		if(b) continue;
		int lt = (p1 == lpos) ? ltype : START_BOUNDARY;
		int rt = (p2 == rpos) ? rtype : END_BOUNDARY;
		double av = 0, d = 1, m = 0;
		if(out.emit) evaluate_rectangle(s, p1, p2, a, e, av, d, m);
		out.push(p1, p2, lt, rt, av, d, m);
	}
	if(rtype == LEFT_SPLICE && !covers_end)
		out.push(rpos - 1, rpos, START_BOUNDARY, rtype, min_weight, 1.0, -1.0);
}

struct graph_params
{
	int min_junction_support;
	int min_subregion_gap, min_subregion_length;
	double min_subregion_overlap, min_guaranteed_edge_weight;
};

KERNEL k_graph_build(const int32_t *order, int n_order, graph_in in, graph_dev g, graph_params prm)
{
	SHARED int s_a, s_b, s_c;
	for(int bi = blockIdx.x; bi < n_order; bi += gridDim.x)
	{
		const int b = order ? order[bi] : bi;
		const int nt = blockDim.x, t = threadIdx.x;
		int32_t *ia = g.iarena + g.iarena_off[b];
		u64 *ka = g.karena + g.karena_off[b];
		const int32_t blpos = in.lpos[b], brpos = in.rpos[b];
		seg_view sv;
		sv.l = in.seg_l + in.seg_off[b]; sv.r = in.seg_r + in.seg_off[b]; sv.c = in.seg_c + in.seg_off[b];
		sv.n = (int)(in.seg_off[b + 1] - in.seg_off[b]);
		const int nh = in.hc.count(b), nf = in.fc.count(b), nch = nh + nf;

		sv.base = in.seg_off[b];
		sv.nhead = in.seg_nhead + sv.base; sv.psum = in.seg_psum + sv.base;

		// ---- junction instances in the order build_junctions feeds jcst: hcst chains, then fcst chains
		int32_t *ci = ia; ia += nch + 1;
		for(int k = t; k < nch; k += nt)
		{
			int len = k < nh ? in.hc.len(b, k) : in.fc.len(b, k - nh);
			ci[k] = (len > 0 && (len & 1) == 0) ? len / 2 : 0;
		}
		BLOCK_SYNC();
		int ninst = block_excl_scan(ci, nch);
		if(t == 0) ci[nch] = ninst;
		BLOCK_SYNC();
		u64 *ikey = ka; ka += ninst + 1;
		u32 *irank = (u32*)ia; ia += ninst + 1;
		for(int k = t; k < nch; k += nt)
		{
			int n2 = ci[k + 1] - ci[k];
			if(n2 <= 0) continue;
			const int32_t *v = k < nh ? in.hc.ptr(b, k) : in.fc.ptr(b, k - nh);
			for(int j = 0; j < n2; j++)
			{
				ikey[ci[k] + j] = ((u64)(u32)v[2 * j] << 32) | (u64)(u32)v[2 * j + 1];
				irank[ci[k] + j] = (u32)(ci[k] + j);
			}
		}
		BLOCK_SYNC();
		block_sort_pairs(ikey, irank, ninst);

		// ---- run-length encode equal (l, r): one junction candidate per run
		int32_t *uhead = ia; ia += ninst + 1;          // exclusive scan of run-head flags -> candidate id
		for(int i = t; i < ninst; i += nt) uhead[i] = (i == 0 || ikey[i] != ikey[i - 1]) ? 1 : 0;
		BLOCK_SYNC();
		int nu = block_excl_scan(uhead, ninst);
		int32_t *u_first = ia; ia += nu + 1;           // first sorted instance of candidate u
		int32_t *u_cnt = ia; ia += 3 * (nu + 1);       // summed AI3
		int32_t *u_lgrp = ia; ia += nu + 1;            // stream rank of the first instance with this lpos
		int32_t *u_keep = ia; ia += nu + 1;
		for(int i = t; i < ninst; i += nt)
			if(i == 0 || ikey[i] != ikey[i - 1]) u_first[uhead[i]] = i;
		if(t == 0) u_first[nu] = ninst;
		BLOCK_SYNC();
		for(int u = t; u < nu; u += nt)
		{
			int a0 = 0, a1 = 0, a2 = 0;
			for(int i = u_first[u]; i < u_first[u + 1]; i++)
			{
				int r = (int)irank[i];
				int k = upper_bound_idx(ci, nch + 1, r) - 1;         // chain of stream position r
				const int32_t *c = k < nh ? in.hc.cnt(b, k) : in.fc.cnt(b, k - nh);
				a0 += c[0]; a1 += c[1]; a2 += c[2];
			}
			u_cnt[3 * u] = a0; u_cnt[3 * u + 1] = a1; u_cnt[3 * u + 2] = a2;
		}
		BLOCK_SYNC();
		// group rank of an lpos = smallest stream rank among candidates sharing it (candidates are sorted by (l, r))
		for(int u = t; u < nu; u += nt)
		{
			u32 l = (u32)(ikey[u_first[u]] >> 32);
			bool head = (u == 0) || ((u32)(ikey[u_first[u - 1]] >> 32) != l);
			if(!head) continue;
			u32 m = 0xffffffffu;
			int e = u;
			while(e < nu && (u32)(ikey[u_first[e]] >> 32) == l) { u32 r = irank[u_first[e]]; if(r < m) m = r; e++; }
			for(int x = u; x < e; x++) u_lgrp[x] = (int32_t)m;
		}
		BLOCK_SYNC();
		// filter (rnacore/graph_builder.cc:93-98) and order by (group rank, own first rank)
		u64 *jkey = ka; ka += nu + 1;
		if(t == 0) s_a = 0;
		BLOCK_SYNC();
		for(int u = t; u < nu; u += nt)
		{
			int32_t l = (int32_t)(u32)(ikey[u_first[u]] >> 32), r = (int32_t)(u32)(ikey[u_first[u]] & 0xffffffffULL);
			int cnt = u_cnt[3 * u] + u_cnt[3 * u + 1] + u_cnt[3 * u + 2];
			int keep = (l < r && cnt >= prm.min_junction_support) ? 1 : 0;
			u_keep[u] = keep;
			if(keep) { int k = atomicAdd(&s_a, 1); jkey[k] = ((u64)(u32)u_lgrp[u] << 32) | (u64)irank[u_first[u]]; }
		}
		BLOCK_SYNC();
		const int nj = s_a;
		block_sort_u64(jkey, nj);
		const int64_t j0 = g.junc_off[b];
		for(int j = t; j < nj; j += nt)
		{
			u32 r = (u32)(jkey[j] & 0xffffffffULL);      // stream rank of the junction's first instance
			int k = upper_bound_idx(ci, nch + 1, (int)r) - 1;
			const int32_t *v = k < nh ? in.hc.ptr(b, k) : in.fc.ptr(b, k - nh);
			int o = (int)r - ci[k];
			int32_t l = v[2 * o], rr = v[2 * o + 1];
			// candidate id by binary search over the sorted unique keys
			u64 key = ((u64)(u32)l << 32) | (u64)(u32)rr;
			int lo = 0, hi = nu;
			while(lo < hi) { int m = (lo + hi) >> 1; if(ikey[u_first[m]] < key) lo = m + 1; else hi = m; }
			int u = lo;
			g.j_l[j0 + j] = l; g.j_r[j0 + j] = rr;
			int a0 = u_cnt[3 * u], a1 = u_cnt[3 * u + 1], a2 = u_cnt[3 * u + 2];
			g.j_cnt[j0 + j] = a0 + a1 + a2;
			g.j_xs0[j0 + j] = a0; g.j_xs1[j0 + j] = a1; g.j_xs2[j0 + j] = a2;
			g.j_strand[j0 + j] = a1 > a2 ? '+' : (a1 < a2 ? '-' : '.');
			g.j_lexon[j0 + j] = -1; g.j_rexon[j0 + j] = -1;
		}
		if(t == 0) g.n_junc[b] = nj;
		BLOCK_SYNC();

		// ---- boundaries (rnacore/graph_builder.cc:177-224): key = pos << 3 | kind, kinds ordered so that the
		// winner of each position comes first: START(0) < END(1) < LEFT(2) < RIGHT(3)
		const int nbk = 2 * nj + 2;
		u64 *bkey = ka; ka += nbk + 1;
		for(int i = t; i < nbk; i += nt)
		{
			u64 k;
			if(i == 0) k = ((u64)(u32)blpos << 3) | 0;
			else if(i == 1) k = ((u64)(u32)brpos << 3) | 1;
			else
			{
				int j = (i - 2) >> 1;
				k = (i & 1) ? (((u64)(u32)g.j_r[j0 + j] << 3) | 3) : (((u64)(u32)g.j_l[j0 + j] << 3) | 2);
			}
			bkey[i] = (k << 24) | (u64)(u32)i;          // make keys distinct
		}
		BLOCK_SYNC();
		block_sort_u64(bkey, nbk);
		int32_t *bflag = ia; ia += nbk + 1;
		for(int i = t; i < nbk; i += nt) bflag[i] = (i == 0 || (bkey[i] >> 27) != (bkey[i - 1] >> 27)) ? 1 : 0;
		BLOCK_SYNC();
		const int nb = block_excl_scan(bflag, nbk);
		int32_t *b_pos = ia; ia += nb + 1;
		int32_t *b_typ = ia; ia += nb + 1;
		for(int i = t; i < nbk; i += nt)
		{
			if(!(i == 0 || (bkey[i] >> 27) != (bkey[i - 1] >> 27))) continue;
			u64 pos = bkey[i] >> 27;
			bool st = false, en = false, le = false, ri = false;
			for(int x = i; x < nbk && (bkey[x] >> 27) == pos; x++)
			{
				int kind = (int)((bkey[x] >> 24) & 7);
				if(kind == 0) st = true; else if(kind == 1) en = true; else if(kind == 2) le = true; else ri = true;
			}
			int ty;
			if(st) ty = START_BOUNDARY;
			else if(en) ty = END_BOUNDARY;
			else if(le && ri) ty = LEFT_RIGHT_SPLICE;
			else if(le) ty = LEFT_SPLICE;
			else ty = RIGHT_SPLICE;
			b_pos[bflag[i]] = (int32_t)(u32)pos;
			b_typ[bflag[i]] = ty;
		}
		BLOCK_SYNC();

		// ---- regions -> partial exons (count, scan, emit)
		const int nreg = nb - 1;
		int32_t *rcnt = ia; ia += nreg + 2;
		const int64_t p0 = g.pex_off[b];
		for(int pass = 0; pass < 2; pass++)
		{
			for(int k = t; k < nreg; k += nt)
			{
				int lt = b_typ[k], rt = b_typ[k + 1];
				if(lt == LEFT_RIGHT_SPLICE) lt = RIGHT_SPLICE;
				if(rt == LEFT_RIGHT_SPLICE) rt = LEFT_SPLICE;
				pexon_sink sink;
				sink.emit = pass; sink.n = 0;
				int64_t o = p0 + (pass ? rcnt[k] : 0);
				sink.l = g.p_l + o; sink.r = g.p_r + o; sink.lt = g.p_lt + o; sink.rt = g.p_rt + o;
				sink.ave = g.p_ave + o; sink.dev = g.p_dev + o; sink.mx = g.p_max + o;
				region_pexons(sv, b_pos[k], b_pos[k + 1], lt, rt, prm.min_subregion_gap, prm.min_subregion_length,
						prm.min_subregion_overlap, prm.min_guaranteed_edge_weight, sink);
				if(!pass) rcnt[k] = sink.n;
			}
			BLOCK_SYNC();
			if(!pass)
			{
				int tot = block_excl_scan(rcnt, nreg);
				if(t == 0) { g.n_pex[b] = tot; s_b = tot; }
				BLOCK_SYNC();
			}
		}
		const int np = s_b;
		BLOCK_SYNC();

		// ---- regional flag + classify (rnacore/graph_builder.cc:226-242, :477-514)
		for(int i = t; i < np; i += nt)
		{
			int32_t l = g.p_l[p0 + i], r = g.p_r[p0 + i];
			int lt = g.p_lt[p0 + i], rt = g.p_rt[p0 + i];
			g.p_regional[p0 + i] = ((l != blpos || r != brpos) && lt == START_BOUNDARY && rt == END_BOUNDARY) ? 1 : 0;
			bool bb = false;
			if(l == blpos) bb = true;
			if(r == brpos) bb = true;
			if(lt == RIGHT_SPLICE) bb = true;
			if(rt == LEFT_SPLICE) bb = true;
			if(lt == LEFT_SPLICE && rt == RIGHT_SPLICE)
			{
				u64 key = ((u64)(u32)l << 32) | (u64)(u32)r;
				int lo = 0, hi = nu;
				while(lo < hi) { int m = (lo + hi) >> 1; if(ikey[u_first[m]] < key) lo = m + 1; else hi = m; }
				bool found = lo < nu && ikey[u_first[lo]] == key && u_keep[lo];
				if(!found) bb = true;
				else if((u_cnt[3 * lo] + u_cnt[3 * lo + 1] + u_cnt[3 * lo + 2]) < g.p_ave[p0 + i]) bb = true;
			}
			g.p_type[p0 + i] = bb ? 0 : 1;             // pvalue 0 -> vertex type 0, pvalue 1 -> type 1
		}
		BLOCK_SYNC();

		// ---- link junctions to partial exons (rnacore/graph_builder.cc:244-297).  The reference asserts that no two partial
		// exons share an lpos or an rpos (:255-258).  Only a 1-bp region between a junction end and a junction start, uncovered
		// and not smoothed (min_subregion_gap 0), breaks that: it gets both stubs, [p, p + 1) twice.  Partial exons are in
		// position order, so such a pair is adjacent; it is reported like a missing exon (AGPU_ERR_INPUT).
		for(int i = t + 1; i < np; i += nt)
			if(g.p_l[p0 + i] == g.p_l[p0 + i - 1] || g.p_r[p0 + i] == g.p_r[p0 + i - 1]) atomicAdd(&g.err[ERR_BOUNDS], 1);
		int32_t *jout = ia; ia += np + 2;              // junction out-degree of pexon i
		int32_t *jin = ia; ia += np + 2;
		for(int i = t; i < np + 2; i += nt) { jout[i] = 0; jin[i] = 0; }
		BLOCK_SYNC();
		for(int j = t; j < nj; j += nt)
		{
			int32_t l = g.j_l[j0 + j], r = g.j_r[j0 + j];
			int le = lower_bound_idx(g.p_r + p0, np, l);
			int re = lower_bound_idx(g.p_l + p0, np, r);
			if(le >= np || g.p_r[p0 + le] != l || re >= np || g.p_l[p0 + re] != r)
			{
				atomicAdd(&g.err[ERR_LINK], 1);          // the reference asserts here
				continue;
			}
			g.j_lexon[j0 + j] = le; g.j_rexon[j0 + j] = re;
			atomicAdd(&jout[le], 1);
			atomicAdd(&jin[re], 1);
		}
		BLOCK_SYNC();

		// ---- vertices (rnacore/graph_builder.cc:305-341)
		const int nv = np + 2;
		const int64_t v0 = vert_base(g, b);
		for(int i = t; i < nv; i += nt)
		{
			if(i == 0 || i == nv - 1)
			{
				int32_t p = (i == 0) ? blpos : brpos;
				g.v_l[v0 + i] = p; g.v_r[v0 + i] = p; g.v_len[v0 + i] = 0; g.v_type[v0 + i] = 0; g.v_regional[v0 + i] = 0;
				g.v_w[v0 + i] = 0; g.v_dev[v0 + i] = 1.0; g.v_max[v0 + i] = 0;
			}
			else
			{
				int k = i - 1;
				double w = g.p_ave[p0 + k];
				if(w < prm.min_guaranteed_edge_weight) w = prm.min_guaranteed_edge_weight;
				g.v_l[v0 + i] = g.p_l[p0 + k]; g.v_r[v0 + i] = g.p_r[p0 + k];
				g.v_len[v0 + i] = g.p_r[p0 + k] - g.p_l[p0 + k];
				g.v_type[v0 + i] = g.p_type[p0 + k]; g.v_regional[v0 + i] = g.p_regional[p0 + k];
				g.v_w[v0 + i] = w; g.v_dev[v0 + i] = g.p_dev[p0 + k]; g.v_max[v0 + i] = g.p_max[p0 + k];
			}
		}

		// ---- edges in insertion order (rnacore/graph_builder.cc:343-423)
		const int64_t e0 = g.edge_off[b];
		int32_t *bcnt = ia; ia += np + 2;              // boundary edges of pexon i (0..2), then scanned
		int32_t *acnt = ia; ia += np + 2;              // adjacency edge after pexon i (0/1), then scanned
		for(int i = t; i < np; i += nt)
		{
			bcnt[i] = (g.p_lt[p0 + i] == START_BOUNDARY ? 1 : 0) + (g.p_rt[p0 + i] == END_BOUNDARY ? 1 : 0);
			acnt[i] = (i + 1 < np && g.p_r[p0 + i] == g.p_l[p0 + i + 1]) ? 1 : 0;
		}
		BLOCK_SYNC();
		// junction edges: junctions with lexon / rexon set, in junction order
		int32_t *jflag = ia; ia += nj + 1;
		for(int j = t; j < nj; j += nt) jflag[j] = (g.j_lexon[j0 + j] >= 0 && g.j_rexon[j0 + j] >= 0) ? 1 : 0;
		BLOCK_SYNC();
		const int nje = block_excl_scan(jflag, nj);
		const int nbe = block_excl_scan(bcnt, np);
		const int nae = block_excl_scan(acnt, np);
		const int ne = nje + nbe + nae;
		for(int j = t; j < nj; j += nt)
		{
			if(g.j_lexon[j0 + j] < 0 || g.j_rexon[j0 + j] < 0) continue;
			int64_t e = e0 + jflag[j];
			g.e_s[e] = g.j_lexon[j0 + j] + 1; g.e_t[e] = g.j_rexon[j0 + j] + 1;
			g.e_w[e] = g.j_cnt[j0 + j];
			g.e_strand[e] = g.j_strand[j0 + j] == '+' ? 1 : (g.j_strand[j0 + j] == '-' ? 2 : 0);
		}
		for(int i = t; i < np; i += nt)
		{
			int64_t e = e0 + nje + bcnt[i];
			double ave = g.p_ave[p0 + i];
			if(g.p_lt[p0 + i] == START_BOUNDARY)
			{
				double w = ave;
				if(i >= 1 && g.p_r[p0 + i - 1] == g.p_l[p0 + i]) w -= g.p_ave[p0 + i - 1];
				if(w < prm.min_guaranteed_edge_weight) w = prm.min_guaranteed_edge_weight;
				g.e_s[e] = 0; g.e_t[e] = i + 1; g.e_w[e] = w; g.e_strand[e] = 0;
				e++;
			}
			if(g.p_rt[p0 + i] == END_BOUNDARY)
			{
				double w = ave;
				if(i < np - 1 && g.p_l[p0 + i + 1] == g.p_r[p0 + i]) w -= g.p_ave[p0 + i + 1];
				if(w < prm.min_guaranteed_edge_weight) w = prm.min_guaranteed_edge_weight;
				g.e_s[e] = i + 1; g.e_t[e] = np + 1; g.e_w[e] = w; g.e_strand[e] = 0;
			}
			if(i + 1 < np && g.p_r[p0 + i] == g.p_l[p0 + i + 1])
			{
				// degrees seen at :404-405 are junction + boundary degrees (see SURVEY appendix C.3)
				int xd = jout[i] + (g.p_rt[p0 + i] == END_BOUNDARY ? 1 : 0);
				int yd = jin[i + 1] + (g.p_lt[p0 + i + 1] == START_BOUNDARY ? 1 : 0);
				double xa = ave, ya = g.p_ave[p0 + i + 1];
				double wt = xa;
				if(xd < yd) wt = xa;
				else if(xd > yd) wt = ya;
				else if(xa < ya) wt = xa;
				else if(xa > ya) wt = ya;
				if(wt < prm.min_guaranteed_edge_weight) wt = prm.min_guaranteed_edge_weight;
				int64_t ea = e0 + nje + nbe + acnt[i];
				g.e_s[ea] = i + 1; g.e_t[ea] = i + 2; g.e_w[ea] = wt; g.e_strand[ea] = 0;
			}
		}
		if(t == 0) g.n_edge[b] = ne;
		BLOCK_SYNC();

		// ---- refine_splice_graph: peel inner vertices with in-degree 0 or out-degree 0 until none is left.
		// The result of this peeling is order independent, so synchronous rounds give the reference's fixed point.
		int32_t *din = ia; ia += nv + 1;
		int32_t *dout = ia; ia += nv + 1;
		int32_t *dead = ia; ia += nv + 1;
		for(int i = t; i < nv; i += nt) { din[i] = 0; dout[i] = 0; dead[i] = 0; }
		BLOCK_SYNC();
		for(int e = t; e < ne; e += nt) { atomicAdd(&dout[g.e_s[e0 + e]], 1); atomicAdd(&din[g.e_t[e0 + e]], 1); }
		BLOCK_SYNC();
		while(true)
		{
			if(t == 0) s_c = 0;
			BLOCK_SYNC();
			for(int i = t + 1; i < nv - 1; i += nt)
			{
				if(dead[i]) continue;
				if(din[i] + dout[i] == 0) continue;
				if(din[i] >= 1 && dout[i] >= 1) continue;
				dead[i] = 1;
				s_c = 1;
			}
			BLOCK_SYNC();
			int any = s_c;
			BLOCK_SYNC();
			if(!any) break;
			for(int e = t; e < ne; e += nt)
			{
				int s = g.e_s[e0 + e];
				if(s < 0) continue;
				int d = g.e_t[e0 + e];
				if(dead[s] == 1 || dead[d] == 1)
				{
					g.e_s[e0 + e] = -1 - s;                // removed: keep the endpoints recoverable
					atomicAdd(&dout[s], -1);
					atomicAdd(&din[d], -1);
				}
			}
			BLOCK_SYNC();
			for(int i = t; i < nv; i += nt) if(dead[i] == 1) dead[i] = 2;
			BLOCK_SYNC();
		}

		// ---- adjacency tables of the refined graph: alive edges sorted by (t, s) and by (s, t)
		u64 *ekey = ka; ka += ne + 1;
		const int64_t vo = voff_base(g, b);
		for(int dir = 0; dir < 2; dir++)
		{
			if(t == 0) s_a = 0;
			BLOCK_SYNC();
			for(int e = t; e < ne; e += nt)
			{
				int s = g.e_s[e0 + e];
				if(s < 0) continue;
				int d = g.e_t[e0 + e];
				int k = atomicAdd(&s_a, 1);
				u64 hi = dir == 0 ? (((u64)(u32)d << 20) | (u64)(u32)s) : (((u64)(u32)s << 20) | (u64)(u32)d);
				ekey[k] = (hi << 24) | (u64)(u32)e;
			}
			BLOCK_SYNC();
			int na = s_a;
			block_sort_u64(ekey, na);
			int32_t *off = (dir == 0 ? g.in_off : g.out_off) + vo;
			int32_t *oth = (dir == 0 ? g.in_src : g.out_dst) + e0;
			int32_t *eid = (dir == 0 ? g.in_eid : g.out_eid) + e0;
			for(int i = t; i <= nv; i += nt) off[i] = 0;
			BLOCK_SYNC();
			for(int k = t; k < na; k += nt)
			{
				int a = (int)((ekey[k] >> 44) & 0xfffff), o = (int)((ekey[k] >> 24) & 0xfffff);
				oth[k] = o;
				eid[k] = (int)(ekey[k] & 0xffffff);
				atomicAdd(&off[a], 1);
			}
			BLOCK_SYNC();
			block_excl_scan(off, nv + 1);
		}
		// prefix count of "breaks": step v -> v + 1 is continuous when the edge exists and the vertices touch
		// (check_continuous_vertices, rnacore/essential.cc:436-446)
		for(int i = t; i < nv; i += nt)
		{
			int brk = 1;
			if(i + 1 < nv && g.v_r[v0 + i] == g.v_l[v0 + i + 1])
			{
				const int32_t *oo = g.out_off + vo;
				for(int k = oo[i]; k < oo[i + 1]; k++) if(g.out_dst[e0 + k] == i + 1) brk = 0;
			}
			g.v_brk[v0 + i] = brk;
		}
		BLOCK_SYNC();
		block_excl_scan(g.v_brk + v0, nv);
		BLOCK_SYNC();
	}
}

} // namespace agpu

#endif
