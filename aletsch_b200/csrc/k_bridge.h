// Stage 4 kernels: bridging of paired-end fragments (bridge/bridge_solver.cc) and
// bundle_base::update_bridges (rnacore/bundle_base.cc:420-507).
//
//   add_adjacent_edges / build_pseudo_introns   :71-108   pseudo edge (i, i+1), weight 0.5, for inner i without one
//   build_bridging_vertices, check_*_relaxing   :53-69, :124-148
//   build_piers / build_bounds                  :150-167, :205-222
//   dynamic_programming / update_stack          :484-546  bottleneck top-K DP, std::sort K-cut (tie order reproduced)
//   nominate / trace_back / refine_pier         :180-274, :548-568
//   vote                                        :276-385
//   helpers: merge_intron_chains (rnacore/essential.cc:474-483), compare/merge_two_sorted_sequences
//   (util/util.h:191-299), check_strand_from_intron_coordinates (rnacore/essential.cc:164-200)
#ifndef ALETSCH_B200_CSRC_K_BRIDGE_H
#define ALETSCH_B200_CSRC_K_BRIDGE_H

#include "runtime.h"
#include "k_cluster.h"

namespace agpu {

#define MAXK AGPU_MAX_DP_SOLUTIONS
#define MAXD AGPU_MAX_DP_STACK

struct sgraph                    // graph of one bundle as the bridge solver sees it (with pseudo edges)
{
	gview gv;
	const int32_t *in_off, *in_src, *in_eid, *out_off, *out_dst, *out_eid;
	const int32_t *e_strand;
	const double *e_w;
	int strand;
};

DEV sgraph sgraph_of(const graph_dev &g, const uint8_t *b_strand, int b)
{
	sgraph s;
	s.gv = graph_of(g, b);
	s.strand = b_strand[b];                 // members of a cluster of bundles share the combined bundle's strand (meta/bundle.cc:93)
	b = graph_index(g, b);
	int64_t vo = voff_base(g, b), e0 = g.edge_off[b];
	s.in_off = g.in_off + vo; s.out_off = g.out_off + vo;
	s.in_src = g.in_src + e0; s.in_eid = g.in_eid + e0; s.out_dst = g.out_dst + e0; s.out_eid = g.out_eid + e0;
	s.e_strand = g.e_strand + e0; s.e_w = g.e_w + e0;
	return s;
}

// real (alive) edge s -> t: index into the bundle's edge arrays, or -1
DEV int real_edge(const sgraph &g, int s, int t)
{
	int lo = g.out_off[s], hi = g.out_off[s + 1];
	int k = lo + lower_bound_idx(g.out_dst + lo, hi - lo, (int32_t)t);
	return (k < hi && g.out_dst[k] == t) ? g.out_eid[k] : -1;
}

// pseudo adjacent edge i -> i + 1 exists iff 1 <= i < nv - 2 and there is no real edge (add_adjacent_edges)
DEV bool pseudo_edge(const sgraph &g, int i) { return i >= 1 && i < g.gv.nv - 2 && real_edge(g, i, i + 1) < 0; }

// gr.edge(s, t) in the solver's graph: 0 none, 1 real (strand in *st), 2 pseudo (strand 0)
DEV int solver_edge(const sgraph &g, int s, int t, int *st)
{
	int e = real_edge(g, s, t);
	if(e >= 0) { *st = g.e_strand[e]; return 1; }
	if(t == s + 1 && pseudo_edge(g, s)) { *st = 0; return 2; }
	return 0;
}

// check_continuous_vertices(gr, x, x + 1) in the solver's graph
DEV bool solver_step_continuous(const sgraph &g, int x)
{
	int st;
	if(!solver_edge(g, x, x + 1, &st)) return false;
	return g.gv.v_r[x] == g.gv.v_l[x + 1];
}

// a sequence made of up to three pieces (chain1 | bridge | chain2, or the pieces of a merge)
struct seq3
{
	const int32_t *p[3];
	int n[3];
	DEV int size() const { return n[0] + n[1] + n[2]; }
	DEV int32_t at(int i) const
	{
		if(i < n[0]) return p[0][i];
		i -= n[0];
		if(i < n[1]) return p[1][i];
		return p[2][i - n[1]];
	}
};

// check_strand_from_intron_coordinates (rnacore/essential.cc:164-200) on the solver's graph
DEV int check_strand(const sgraph &g, const seq3 &w)
{
	int n = w.size() / 2;
	if(n <= 0) return 0;
	bool b1 = false, b2 = false;
	for(int k = 0; k < n; k++)
	{
		int32_t p = w.at(2 * k), q = w.at(2 * k + 1);
		if(p >= q) return -1;
		int kp = rindex_find(g.gv, p), kq = lindex_find(g.gv, q);
		if(kp < 0 || kq < 0) return -1;
		int st = 0;
		if(!solver_edge(g, kp, kq, &st)) return -1;
		if(st == 1) b1 = true;
		if(st == 2) b2 = true;
	}
	if(b1 && b2) return -1;
	if(b1) return 1;
	if(b2) return 2;
	return 0;
}

DEV bool seq_increasing(const seq3 &w)
{
	int n = w.size();
	for(int k = 0; k + 1 < n; k++) if(w.at(k) > w.at(k + 1)) return false;
	return true;
}

// positions as in util/constants.h:66-76
enum { IDENTICAL = 0, FALL_RIGHT, FALL_LEFT, CONTAINED, CONTAINING, EXTEND_RIGHT, EXTEND_LEFT, NESTED, NESTING, CONFLICTING };

DEV bool check_identical(const int32_t *x, int x1, int x2, const int32_t *y, int y1, int y2)
{
	if(x[x1] != y[y1]) return false;
	if(x[x2] != y[y2]) return false;
	if(x2 - x1 != y2 - y1) return false;
	for(int kx = x1, ky = y1; kx <= x2 && ky <= y2; kx++, ky++) if(x[kx] != y[ky]) return false;
	return true;
}

// compare_two_sorted_sequences (util/util.h:191-253); both sequences non-empty
DEV int compare_sorted(const int32_t *ref, int nr, const int32_t *qry, int nq)
{
	if(ref[nr - 1] < qry[0]) return FALL_RIGHT;
	if(ref[0] > qry[nq - 1]) return FALL_LEFT;
	int kr1 = lower_bound_idx(ref, nr, qry[0]);
	int kq1 = lower_bound_idx(qry, nq, ref[0]);
	int kq2 = lower_bound_idx(qry, nq, ref[nr - 1]);
	int kr2 = lower_bound_idx(ref, nr, qry[nq - 1]);
	bool r2end = kr2 >= nr, q2end = kq2 >= nq;
	if(kr1 >= nr || kq1 >= nq) return CONFLICTING;     // the reference asserts these away
	if(qry[kq1] == ref[0] || ref[kr1] == qry[0])
	{
		if(!r2end && !q2end)
		{
			bool b = check_identical(ref, kr1, kr2, qry, kq1, kq2);
			if(!b) return CONFLICTING;
			if(kr1 == 0 && kq1 == 0) return IDENTICAL;
			if(kr1 >= 1 && kq1 == 0) return CONTAINED;
			if(kr1 == 0 && kq1 >= 1) return CONTAINING;
			return CONFLICTING;
		}
		else if(!r2end && q2end)
		{
			bool b = check_identical(ref, kr1, kr2, qry, kq1, nq - 1);
			if(!b) return CONFLICTING;
			if(kq1 == 0) return CONTAINED;
			return EXTEND_LEFT;
		}
		else if(r2end && !q2end)
		{
			bool b = check_identical(ref, kr1, nr - 1, qry, kq1, kq2);
			if(!b) return CONFLICTING;
			if(kr1 == 0) return CONTAINING;
			return EXTEND_RIGHT;
		}
	}
	else if(ref[kr1] > qry[0] && kr2 == kr1 && ref[kr2] > qry[nq - 1]) return NESTED;
	else if(qry[kq1] > ref[0] && kq2 == kq1 && qry[kq2] > ref[nr - 1]) return NESTING;
	return CONFLICTING;
}

// merge_intron_chains(x, y, xy) (rnacore/essential.cc:474-483) with xy returned as pieces
DEV bool merge_intron_chains(const int32_t *x, int nx, const int32_t *y, int ny, seq3 &xy)
{
	xy.n[0] = xy.n[1] = xy.n[2] = 0;
	xy.p[0] = xy.p[1] = xy.p[2] = x;
	if(nx >= 1 && ny >= 1 && x[0] > y[0]) return false;
	if(nx == 0) { xy.p[0] = y; xy.n[0] = ny; }
	else if(ny == 0) { xy.p[0] = x; xy.n[0] = nx; }
	else
	{
		int t = compare_sorted(x, nx, y, ny);
		if(t == CONFLICTING || t == NESTED || t == NESTING) return false;
		if(t == IDENTICAL || t == CONTAINED) { xy.p[0] = x; xy.n[0] = nx; }
		if(t == CONTAINING) { xy.p[0] = y; xy.n[0] = ny; }
		if(t == FALL_RIGHT) { xy.p[0] = x; xy.n[0] = nx; xy.p[1] = y; xy.n[1] = ny; }
		if(t == FALL_LEFT) { xy.p[0] = y; xy.n[0] = ny; xy.p[1] = x; xy.n[1] = nx; }
		if(t == EXTEND_LEFT)
		{
			int q1 = lower_bound_idx(y, ny, x[0]);
			xy.p[0] = y; xy.n[0] = q1; xy.p[1] = x; xy.n[1] = nx;
		}
		if(t == EXTEND_RIGHT)
		{
			int q2 = lower_bound_idx(y, ny, x[nx - 1]);
			xy.p[0] = x; xy.n[0] = nx; xy.p[1] = y + q2 + 1; xy.n[1] = ny - q2 - 1;
		}
	}
	int d = nx + ny - xy.size();
	if(d % 2 != 0) return false;
	return true;
}

struct bridge_dev
{
	int K, D;
	int relax, low, high;
	// per cluster
	int32_t *vp1, *vp2;
	int32_t *pier_of;            // pier index (global) of the cluster, -1
	// piers: scratch at clu_off[b] + k, sorted by (bs, bt) within the bundle
	int32_t *n_piers, *n_groups;
	int32_t *p_bs, *p_bt;
	int32_t *p_group;            // group (global job base) of the pier
	// pier groups (DP jobs): at clu_off[b] + j
	int32_t *g_k1, *g_k2, *g_first, *g_last;   // vertex range, pier range (bundle-local pier indices)
	int64_t *g_rows;             // rows needed: (k2 - k1 + 1) * passes  -> scanned into g_row_off
	int64_t *g_row_off;
	int32_t *maxin;              // [NB] max in-degree (+1 for the pseudo edge)
	// DP tables: row r holds up to K entries
	int32_t *t_cnt, *t_len, *t_tr1, *t_tr2, *t_stack;
	// candidate scratch per job
	int64_t *g_cand_off;
	int32_t *cand;               // per candidate: D stack ints, len, tr1, tr2
	int32_t *cand_idx;
	// bridges per pier
	int64_t *p_path_off;         // scanned: room for 2K paths of (bt - bs + 1) vertices + chains of twice that
	int32_t *p_nbr;
	int32_t *br_len, *br_clen, *br_stack;      // per pier slot (2K slots): path length, chain length, stack
	int32_t *br_order;           // [2K per pier] order after refine_pier
	int32_t *paths, *chains;
};

HD int passes_of(int strand) { return strand == '.' ? 2 : ((strand == '+' || strand == '-') ? 1 : 0); }
HD int pass_strand(int strand, int k) { return strand == '.' ? k + 1 : (strand == '+' ? 1 : 2); }

// ---- B1: bridging vertices of every cluster (build_bridging_vertices)
KERNEL k_bridge_vertices(int64_t n_clu, const int32_t *c_bundle, const int32_t *c_bounds, const int32_t *c_chain1, const int32_t *c_chain2,
		chains_view cv, graph_dev g, const uint8_t *b_strand, bridge_dev br)
{
	int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(c >= n_clu) return;
	int b = c_bundle[c];
	sgraph sg = sgraph_of(g, b_strand, b);
	const gview &gv = sg.gv;
	int n = gv.nv - 1;
	int32_t bd1 = c_bounds[4 * c + 1], bd2 = c_bounds[4 * c + 2];
	int v1 = locate_vertex(gv, bd1 - 1);
	int v2 = locate_vertex(gv, bd2);
	// check_left_relaxing
	{
		int v = v1;
		bool ok = !(v <= 0 || v >= n);
		if(ok && v <= 1) ok = false;
		if(ok && !solver_step_continuous(sg, v - 1)) ok = false;
		if(ok && bd1 - gv.v_l[v] > br.relax) ok = false;
		if(ok && c_chain1[c] >= 0)
		{
			int len = cv.len(b, c_chain1[c]);
			if(len >= 1 && cv.ptr(b, c_chain1[c])[len - 1] >= gv.v_l[v]) ok = false;
		}
		if(ok) v1--;
	}
	{
		int v = v2;
		bool ok = !(v <= 0 || v >= n);
		if(ok && v >= n - 1) ok = false;
		if(ok && !solver_step_continuous(sg, v)) ok = false;
		if(ok && gv.v_r[v] - bd2 > br.relax) ok = false;
		if(ok && c_chain2[c] >= 0)
		{
			int len = cv.len(b, c_chain2[c]);
			if(len >= 1 && cv.ptr(b, c_chain2[c])[0] <= gv.v_r[v]) ok = false;
		}
		if(ok) v2++;
	}
	br.vp1[c] = v1; br.vp2[c] = v2;
}

// ---- B2: piers and pier groups of every bundle (build_piers, build_bounds); one CTA per bundle
KERNEL k_piers(const int32_t *order, int32_t n_bundles, const int64_t *clu_off, graph_dev g, const uint8_t *b_strand, bridge_dev br, u64 *key_scratch)
{
	SHARED int s_n, s_max;
	for(int bi = blockIdx.x; bi < n_bundles; bi += gridDim.x)
	{
		const int b = order ? order[bi] : bi;
		int64_t c0 = clu_off[b];
		int nc = (int)(clu_off[b + 1] - c0);
		u64 *key = key_scratch + c0;
		if(threadIdx.x == 0) { s_n = 0; s_max = 0; }
		BLOCK_SYNC();
		for(int c = threadIdx.x; c < nc; c += blockDim.x)
		{
			int v1 = br.vp1[c0 + c], v2 = br.vp2[c0 + c];
			if(v1 < 0 || v2 < 0 || v1 >= v2) continue;
			int k = atomicAdd(&s_n, 1);
			key[k] = ((u64)(u32)v1 << 32) | (u64)(u32)v2;
		}
		// largest in-degree, for the candidate scratch of the DP
		if(graph_index(g, b) >= 0)
		{
			const int gb = graph_index(g, b);
			int nv = g.n_pex[gb] + 2;
			const int32_t *io = g.in_off + voff_base(g, gb);
			int m = 0;
			for(int v = threadIdx.x; v < nv; v += blockDim.x) { int d = io[v + 1] - io[v]; if(d > m) m = d; }
			atomicMax(&s_max, m);
		}
		BLOCK_SYNC();
		int n = s_n;
		// sort + unique; equal keys are harmless for the network (swapping equal values is invisible)
		block_sort_u64(key, n);
		int32_t *flag = br.p_group + c0;      // reused as scratch until the groups are known
		for(int i = threadIdx.x; i < n; i += blockDim.x) flag[i] = (i == 0 || key[i] != key[i - 1]) ? 1 : 0;
		BLOCK_SYNC();
		int np = block_excl_scan(flag, n);
		for(int i = threadIdx.x; i < n; i += blockDim.x)
			if(i == 0 || key[i] != key[i - 1]) { br.p_bs[c0 + flag[i]] = (int32_t)(key[i] >> 32); br.p_bt[c0 + flag[i]] = (int32_t)(u32)(key[i] & 0xffffffffULL); }
		BLOCK_SYNC();
		// groups: runs of equal bs
		for(int i = threadIdx.x; i < np; i += blockDim.x) flag[i] = (i == 0 || br.p_bs[c0 + i] != br.p_bs[c0 + i - 1]) ? 1 : 0;
		BLOCK_SYNC();
		int ng = block_excl_scan(flag, np);
		int passes = passes_of(b_strand[b]);
		for(int i = threadIdx.x; i < np; i += blockDim.x)
		{
			bool head = (i == 0 || br.p_bs[c0 + i] != br.p_bs[c0 + i - 1]);
			if(!head) continue;
			int j = i;
			while(j + 1 < np && br.p_bs[c0 + j + 1] == br.p_bs[c0 + i]) j++;
			int gi = flag[i];
			br.g_k1[c0 + gi] = br.p_bs[c0 + i];
			br.g_k2[c0 + gi] = br.p_bt[c0 + j];          // farthest target: piers are sorted by (bs, bt)
			br.g_first[c0 + gi] = i; br.g_last[c0 + gi] = j;
			br.g_rows[c0 + gi] = (int64_t)(br.p_bt[c0 + j] - br.p_bs[c0 + i] + 1) * passes;
		}
		BLOCK_SYNC();
		for(int i = threadIdx.x; i < np; i += blockDim.x)
		{
			// group of pier i = number of heads at or before i, minus one
			int head = (i == 0 || br.p_bs[c0 + i] != br.p_bs[c0 + i - 1]) ? 1 : 0;
			br.p_nbr[c0 + i] = flag[i] + head - 1;     // temporarily: the pier's group index
		}
		BLOCK_SYNC();
		for(int i = threadIdx.x; i < np; i += blockDim.x) br.p_group[c0 + i] = br.p_nbr[c0 + i];
		for(int i = threadIdx.x; i < nc; i += blockDim.x) if(i >= ng) br.g_rows[c0 + i] = 0;
		BLOCK_SYNC();
		for(int i = threadIdx.x; i < np; i += blockDim.x)
		{
			br.p_nbr[c0 + i] = 0;
			br.p_path_off[c0 + i] = (int64_t)2 * br.K * (br.p_bt[c0 + i] - br.p_bs[c0 + i] + 1);
		}
		for(int i = threadIdx.x; i < nc; i += blockDim.x) if(i >= np) br.p_path_off[c0 + i] = 0;
		if(threadIdx.x == 0) { br.n_piers[b] = np; br.n_groups[b] = ng; br.maxin[b] = s_max + 1; }
		BLOCK_SYNC();
	}
}

// pier index of every cluster
KERNEL k_cluster_pier(int64_t n_clu, const int32_t *c_bundle, const int64_t *clu_off, bridge_dev br)
{
	int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(c >= n_clu) return;
	br.pier_of[c] = -1;
	int v1 = br.vp1[c], v2 = br.vp2[c];
	if(v1 < 0 || v2 < 0 || v1 >= v2) return;
	int b = c_bundle[c];
	int64_t c0 = clu_off[b];
	int np = br.n_piers[b];
	int lo = 0, hi = np;
	while(lo < hi)
	{
		int m = (lo + hi) >> 1;
		int bs = br.p_bs[c0 + m], bt = br.p_bt[c0 + m];
		if(bs < v1 || (bs == v1 && bt < v2)) lo = m + 1; else hi = m;
	}
	if(lo < np && br.p_bs[c0 + lo] == v1 && br.p_bt[c0 + lo] == v2) br.pier_of[c] = lo;
}

// candidate scratch of every group: (max in-degree + 1) * K entries for each of the two strand passes
KERNEL k_group_cand(int64_t n_slots, int32_t n_bundles, const int64_t *clu_off, bridge_dev br, int64_t *cand_need)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_slots) return;
	int b = find_segment(clu_off, n_bundles, i);
	int gi = (int)(i - clu_off[b]);
	cand_need[i] = gi < br.n_groups[b] ? (int64_t)2 * br.maxin[b] * br.K : 0;       // one stretch per strand pass: the passes run side by side
}

struct entry_less
{
	const int32_t *cand;
	int D, W;
	// entry_compare (bridge/bridge_solver.cc:21-30)
	HD bool operator()(int x, int y) const
	{
		const int32_t *a = cand + (int64_t)x * W, *b = cand + (int64_t)y * W;
		for(int i = 0; i < D; i++)
		{
			if(a[i] > b[i]) return true;
			if(a[i] < b[i]) return false;
		}
		return a[D] < b[D];
	}
};

// dense work lists of the bridging kernels: DP jobs = (pier group, strand pass), trace-back jobs = piers
KERNEL k_bridge_job_counts(int64_t nb, const uint8_t *b_strand, bridge_dev br, int64_t *n_dp, int64_t *n_pier)
{
	int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(b >= nb) return;
	n_dp[b] = (int64_t)br.n_groups[b] * passes_of(b_strand[b]);
	n_pier[b] = br.n_piers[b];
}

KERNEL k_bridge_job_fill(int64_t nb, const int64_t *clu_off, const uint8_t *b_strand, bridge_dev br, const int64_t *dp_off, const int64_t *pier_off,
		int64_t *dp_job, int32_t *dp_bundle, int64_t *pier_job, int32_t *pier_bundle)
{
	int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(b >= nb) return;
	int np = passes_of(b_strand[b]);
	int64_t o = dp_off[b];
	for(int gi = 0; gi < br.n_groups[b]; gi++)
		for(int pass = 0; pass < np; pass++) { dp_job[o] = ((clu_off[b] + gi) << 1) | pass; dp_bundle[o] = (int32_t)b; o++; }
	o = pier_off[b];
	for(int pi = 0; pi < br.n_piers[b]; pi++) { pier_job[o] = clu_off[b] + pi; pier_bundle[o] = (int32_t)b; o++; }
}

// ---- B3: bottleneck top-K DP (dynamic_programming, bridge/bridge_solver.cc:484-530 with update_stack :532-546), one WARP per
// (pier group, strand pass).  Per vertex the warp's lanes take the
// in-edges (coalesced reads of the CSR row), a warp scan places every edge's candidates, the lanes then build the candidates
// -- update_stack of one predecessor entry each -- into the warp's shared-memory slice, and rank them by counting under
// entry_compare (rank = number of smaller candidates + number of equal ones generated earlier: the stable order).  std::sort of
// the reference is stable for up to 16 elements (pure insertion sort) and, whatever its internals, yields THE sorted order when
// no two candidates compare equal; only a vertex with more than 16 candidates AND a tie is handed to one lane for the exact
// libstdc++ replay (stdsort.h), on the shared-memory copy.  The K best go to the table row in global memory (the trace-back
// needs every row), written by the lanes that own them.
#ifndef AGPU_EMU
#define DPW_WS 32
#else
#define DPW_WS 1                 // kernel-logic build: a "warp" of one lane runs the same code
#endif
#define DPW_WARPS 4              // warps per CTA
#define DPW_CMAX 128             // candidates per vertex kept in shared memory (more: the job falls back to the scratch in global memory)
#define DPW_EMAX 64              // in-edges per vertex kept in shared memory
#define DPW_W (AGPU_MAX_DP_STACK + 3)

DEV int dpw_excl_scan(int v, int lane, int *total)
{
#ifndef AGPU_EMU
	int inc = v;
#pragma unroll
	for(int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, inc, o); if(lane >= o) inc += y; }
	*total = __shfl_sync(0xffffffffu, inc, 31);
	return inc - v;
#else
	(void)lane;
	*total = v;
	return 0;
#endif
}
DEV void dpw_sync()
{
#ifndef AGPU_EMU
	__syncwarp();
#endif
}
DEV int dpw_any(int p)
{
#ifndef AGPU_EMU
	return __any_sync(0xffffffffu, p);
#else
	return p;
#endif
}

// a < b under entry_compare (bridge/bridge_solver.cc:21-30) on shared-memory candidates of stride DPW_W
DEV int dpw_cmp(const int32_t *a, const int32_t *b, int D)
{
	for(int i = 0; i < D; i++)
	{
		if(a[i] > b[i]) return -1;
		if(a[i] < b[i]) return 1;
	}
	if(a[D] < b[D]) return -1;
	if(a[D] > b[D]) return 1;
	return 0;
}

KERNEL k_bridge_dp_warp(int64_t n_jobs, const int64_t *dp_job, const int32_t *dp_bundle, const int64_t *clu_off, graph_dev g, const uint8_t *b_strand,
		bridge_dev br)
{
	SHARED int32_t s_cand[DPW_WARPS][DPW_CMAX * DPW_W];
	SHARED int32_t s_rank[DPW_WARPS][DPW_CMAX];
	SHARED int32_t s_ej[DPW_WARPS][DPW_EMAX], s_ew[DPW_WARPS][DPW_EMAX], s_eo[DPW_WARPS][DPW_EMAX + 1];
	const int WS = DPW_WS;
	const int lane = threadIdx.x % WS, wid = threadIdx.x / WS, wpc = blockDim.x / WS > 0 ? blockDim.x / WS : 1;
	int32_t *cand = s_cand[wid], *rank = s_rank[wid], *ej = s_ej[wid], *ew = s_ew[wid], *eo = s_eo[wid];
	for(int64_t ji = (int64_t)blockIdx.x * wpc + wid; ji < n_jobs; ji += (int64_t)gridDim.x * wpc)
	{
		const int64_t job = dp_job[ji];
		const int64_t slot = job >> 1;
		const int pass = (int)(job & 1);
		const int b = dp_bundle[ji];
		const sgraph sg = sgraph_of(g, b_strand, b);
		const int strand = pass_strand(sg.strand, pass);
		const int K = br.K, D = br.D, W = D + 3;
		const int k1 = br.g_k1[slot], k2 = br.g_k2[slot];
		const int nrow = k2 - k1 + 1;
		const int64_t row0 = br.g_row_off[slot] + (int64_t)pass * nrow;
		const int64_t poff = (int64_t)pass * br.maxin[b] * K;
		int32_t *gcand = br.cand + (br.g_cand_off[slot] + poff) * W;
		int32_t *gcidx = br.cand_idx + br.g_cand_off[slot] + poff;
		if(lane == 0)
		{
			// table[k1]: one entry, stack of D times 999999, length of the vertex, no trace
			br.t_cnt[row0] = 1;
			for(int d = 0; d < D; d++) br.t_stack[row0 * K * D + d] = 999999;
			br.t_len[row0 * K] = sg.gv.v_r[k1] - sg.gv.v_l[k1];
			br.t_tr1[row0 * K] = -1; br.t_tr2[row0 * K] = -1;
		}
		dpw_sync();
		for(int k = k1 + 1; k <= k2; k++)
		{
			const int64_t row = row0 + (k - k1);
			const int32_t len = sg.gv.v_r[k] - sg.gv.v_l[k];
			const int lo = sg.in_off[k], hi = sg.in_off[k + 1];
			const int ne = hi - lo + (pseudo_edge(sg, k - 1) ? 1 : 0);
			if(ne > DPW_EMAX)
			{
				// more in-edges than the shared slice holds: the sequential form of the reference on the global scratch (one lane)
				if(lane == 0)
				{
					int nc = 0;
					for(int x = lo; x < lo + ne; x++)
					{
						int j, w, s;
						if(x < hi) { int e = sg.in_eid[x]; j = sg.in_src[x]; s = sg.e_strand[e]; w = (int)sg.e_w[e]; }
						else { j = k - 1; s = 0; w = 0; }
						if(s != 0 && s != strand) continue;
						if(j < k1) continue;
						const int64_t jr = row0 + (j - k1);
						const int nj = br.t_cnt[jr];
						for(int i = 0; i < nj; i++)
						{
							int32_t *ce = gcand + (int64_t)nc * W;
							const int32_t *v = br.t_stack + (jr * K + i) * D;
							for(int q = 0; q < D; q++) ce[q] = 0;
							for(int a = 0, q = 0; a < D && q < D; a++, q++)
							{
								if(a == q && v[a] > w) { ce[q] = w; q++; if(q >= D) break; }
								ce[q] = v[a];
							}
							ce[D] = br.t_len[jr * K + i] + len; ce[D + 1] = j; ce[D + 2] = i;
							gcidx[nc] = nc;
							nc++;
						}
					}
					entry_less less;
					less.cand = gcand; less.D = D; less.W = W;
					std_sort_handles(gcidx, nc, less);
					const int keep = nc > K ? K : nc;
					br.t_cnt[row] = keep;
					for(int i = 0; i < keep; i++)
					{
						const int32_t *ce = gcand + (int64_t)gcidx[i] * W;
						for(int d = 0; d < D; d++) br.t_stack[(row * K + i) * D + d] = ce[d];
						br.t_len[row * K + i] = ce[D]; br.t_tr1[row * K + i] = ce[D + 1]; br.t_tr2[row * K + i] = ce[D + 2];
					}
				}
				dpw_sync();
				continue;
			}
			// in-edges in (source, target) order; the pseudo edge from k - 1, if any, has the largest source
			int carry = 0;
			for(int x0 = 0; x0 < ne; x0 += WS)
			{
				const int x = x0 + lane;
				int j = -1, w = 0, nj = 0;
				if(x < ne)
				{
					int s;
					if(lo + x < hi) { const int e = sg.in_eid[lo + x]; j = sg.in_src[lo + x]; s = sg.e_strand[e]; w = (int)sg.e_w[e]; }
					else { j = k - 1; s = 0; w = 0; }            // (int)0.5
					if((s == 0 || s == strand) && j >= k1) nj = br.t_cnt[row0 + (j - k1)];
				}
				int tot;
				const int off = carry + dpw_excl_scan(nj, lane, &tot);
				if(x < ne) { ej[x] = j; ew[x] = w; eo[x] = off; }
				carry += tot;
			}
			if(lane == 0) eo[ne] = carry;
			const int nc = carry;
			dpw_sync();
			const bool in_smem = nc <= DPW_CMAX;
			int32_t *cd = in_smem ? cand : gcand;
			const int CW = in_smem ? DPW_W : W;
			for(int c = lane; c < nc; c += WS)
			{
				// edge of candidate c: last e with eo[e] <= c
				int e = 0;
				{
					int a = 0, z = ne;
					while(a < z) { int m = (a + z) >> 1; if(eo[m + 1] <= c) a = m + 1; else z = m; }
					e = a;
				}
				const int j = ej[e], w = ew[e], i = c - eo[e];
				const int64_t jr = row0 + (j - k1);
				int32_t *ce = cd + (int64_t)c * CW;
				const int32_t *v = br.t_stack + (jr * K + i) * D;
				// update_stack (:532-546)
				for(int q = 0; q < D; q++) ce[q] = 0;
				for(int a = 0, q = 0; a < D && q < D; a++, q++)
				{
					if(a == q && v[a] > w) { ce[q] = w; q++; if(q >= D) break; }
					ce[q] = v[a];
				}
				ce[D] = br.t_len[jr * K + i] + len; ce[D + 1] = j; ce[D + 2] = i;
			}
			dpw_sync();
			const int keep = nc > K ? K : nc;
			if(in_smem)
			{
				int tie = 0;
				for(int c = lane; c < nc; c += WS)
				{
					const int32_t *me = cd + c * CW;
					int r = 0;
					for(int o = 0; o < nc; o++)
					{
						if(o == c) continue;
						const int q = dpw_cmp(cd + o * CW, me, D);
						if(q < 0 || (q == 0 && o < c)) r++;
						if(q == 0) tie = 1;
					}
					rank[c] = r;
				}
				if(nc > 16 && dpw_any(tie))
				{
					// more than 16 candidates with a tie: the reference's introsort decides the order of the equal ones
					dpw_sync();
					if(lane == 0)
					{
						int32_t *idx = gcidx;
						for(int c = 0; c < nc; c++) idx[c] = c;
						entry_less less;
						less.cand = cd; less.D = D; less.W = CW;
						std_sort_handles(idx, nc, less);
						for(int r = 0; r < nc; r++) rank[idx[r]] = r;
					}
					dpw_sync();
				}
				for(int c = lane; c < nc; c += WS)
				{
					const int r = rank[c];
					if(r >= keep) continue;
					const int32_t *ce = cd + c * CW;
					for(int d = 0; d < D; d++) br.t_stack[(row * K + r) * D + d] = ce[d];
					br.t_len[row * K + r] = ce[D]; br.t_tr1[row * K + r] = ce[D + 1]; br.t_tr2[row * K + r] = ce[D + 2];
				}
			}
			else if(lane == 0)
			{
				for(int c = 0; c < nc; c++) gcidx[c] = c;
				entry_less less;
				less.cand = cd; less.D = D; less.W = CW;
				std_sort_handles(gcidx, nc, less);
				for(int i = 0; i < keep; i++)
				{
					const int32_t *ce = cd + (int64_t)gcidx[i] * CW;
					for(int d = 0; d < D; d++) br.t_stack[(row * K + i) * D + d] = ce[d];
					br.t_len[row * K + i] = ce[D]; br.t_tr1[row * K + i] = ce[D + 1]; br.t_tr2[row * K + i] = ce[D + 2];
				}
			}
			if(lane == 0) br.t_cnt[row] = keep;
			dpw_sync();
		}
	}
}

struct path_less               // compare_bridge_path_vertices (bridge/bridge_path.cc:58-68)
{
	const int32_t *paths, *len;
	int stride;
	HD bool operator()(int x, int y) const
	{
		const int32_t *a = paths + (int64_t)x * stride, *b = paths + (int64_t)y * stride;
		int na = len[x], nb = len[y];
		for(int k = 0; k < na && k < nb; k++)
		{
			if(a[k] < b[k]) return true;
			if(a[k] > b[k]) return false;
		}
		return na < nb;
	}
};

struct stack_greater           // compare_bridge_path_stack (bridge/bridge_path.cc:76-84); stacks have equal sizes
{
	const int32_t *stack;
	int D;
	HD bool operator()(int x, int y) const
	{
		const int32_t *a = stack + (int64_t)x * D, *b = stack + (int64_t)y * D;
		for(int k = 0; k < D; k++)
		{
			if(a[k] > b[k]) return true;
			if(a[k] < b[k]) return false;
		}
		return false;
	}
};

// ---- B4: trace back, build the candidate bridges of every pier and order them (nominate :224-257, refine_pier :259-274)
KERNEL_OCC(6) k_pier_bridges(int64_t n_jobs, const int64_t *pier_job, const int32_t *pier_bundle, const int64_t *clu_off, graph_dev g,
		const uint8_t *b_strand, bridge_dev br)
{
	int64_t ji = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(ji >= n_jobs) return;
	int64_t slot = pier_job[ji];
	int b = pier_bundle[ji];
	int64_t c0 = clu_off[b];
	sgraph sg = sgraph_of(g, b_strand, b);
	const int K = br.K, D = br.D;
	int bs = br.p_bs[slot], bt = br.p_bt[slot];
	int stride = bt - bs + 1;
	int64_t gslot = c0 + br.p_group[slot];
	int k1 = br.g_k1[gslot], k2 = br.g_k2[gslot];
	int nrow = k2 - k1 + 1;
	int32_t *paths = br.paths + br.p_path_off[slot];
	int32_t *chains = br.chains + 2 * br.p_path_off[slot];
	int32_t *blen = br.br_len + slot * 2 * K, *bclen = br.br_clen + slot * 2 * K, *bstack = br.br_stack + slot * 2 * K * D;
	int32_t *order = br.br_order + slot * 2 * K;
	int nb = 0;
	int np = passes_of(sg.strand);
	for(int pass = 0; pass < np; pass++)
	{
		int64_t row = br.g_row_off[gslot] + (int64_t)pass * nrow + (bt - k1);
		int cnt = br.t_cnt[row];
		for(int i = 0; i < cnt; i++)
		{
			// trace_back: vertices from bt back to k1, then reversed
			int32_t *pv = paths + (int64_t)nb * stride;
			int n = 0;
			int p = bt, q = i;
			while(true)
			{
				pv[n++] = p;
				int64_t r = br.g_row_off[gslot] + (int64_t)pass * nrow + (p - k1);
				int np1 = br.t_tr1[r * K + q], nq = br.t_tr2[r * K + q];
				p = np1; q = nq;
				if(p < 0) break;
			}
			for(int x = 0, y = n - 1; x < y; x++, y--) { int32_t t = pv[x]; pv[x] = pv[y]; pv[y] = t; }
			blen[nb] = n;
			for(int d = 0; d < D; d++) bstack[nb * D + d] = br.t_stack[(row * K + i) * D + d];
			// intron coordinates of the path without pseudo introns (build_intron_coordinates_from_path + filter_pseudo_introns)
			int32_t *cv = chains + (int64_t)nb * 2 * stride;
			int cl = 0;
			for(int x = 0; x + 1 < n; x++)
			{
				int32_t pp = sg.gv.v_r[pv[x]], qq = sg.gv.v_l[pv[x + 1]];
				if(pp == qq) continue;
				if(pv[x + 1] == pv[x] + 1 && pseudo_edge(sg, pv[x])) continue;
				cv[cl++] = pp; cv[cl++] = qq;
			}
			bclen[nb] = cl;
			order[nb] = nb;
			nb++;
		}
	}
	// refine_pier
	int m = nb;
	if(nb > 0)
	{
		path_less pl;
		pl.paths = paths; pl.len = blen; pl.stride = stride;
		std_sort_handles(order, nb, pl);
		m = 1;
		for(int i = 1; i < nb; i++)
		{
			int a = order[i], c = order[i - 1];
			bool same = blen[a] == blen[c];
			for(int k = 0; same && k < blen[a]; k++) if(paths[(int64_t)a * stride + k] != paths[(int64_t)c * stride + k]) same = false;
			if(same) continue;
			order[m++] = order[i];
		}
		stack_greater sgt;
		sgt.stack = bstack; sgt.D = D;
		std_sort_handles(order, m, sgt);
	}
	br.p_nbr[slot] = m;
}

// ---- B5: vote (bridge/bridge_solver.cc:287-385)
//   k_vote (emit = 0)  one thread per cluster: classify; clusters without a decision to take are settled at once, the
//                      others are packed into two work lists (any order: results are addressed by cluster)
//   k_vote_type1       one thread per listed cluster with overlapping end vertices: merge the two chains, one candidate
//   k_vote_type2       one thread per listed cluster with a pier: the bridge candidates in refine_pier order, the first valid
//                      one is the choice (a warp per cluster was measured slower: most piers offer 1-3 candidates)
//   k_vote (emit = 1)  one thread per cluster writes the coordinates of the chosen chain / whole
struct vote_lists { int32_t *n1, *list1, *n2, *list2; };

struct vote_cluster              // what every vote kernel needs about a cluster
{
	int b, type, n1, n2;
	int64_t slot;
	const int32_t *ch1, *ch2;
};

DEV vote_cluster vote_load(int64_t c, int ss, int tt, const int32_t *c_bundle, const int64_t *clu_off, const int32_t *c_chain1,
		const int32_t *c_chain2, const chains_view &cv, const bridge_dev &br)
{
	vote_cluster v;
	v.b = c_bundle[c];
	v.ch1 = NULL; v.ch2 = NULL; v.n1 = 0; v.n2 = 0;
	if(c_chain1[c] >= 0) { v.ch1 = cv.ptr(v.b, c_chain1[c]); v.n1 = cv.len(v.b, c_chain1[c]); }
	if(c_chain2[c] >= 0) { v.ch2 = cv.ptr(v.b, c_chain2[c]); v.n2 = cv.len(v.b, c_chain2[c]); }
	v.type = 0; v.slot = -1;
	if(ss >= tt) v.type = 1;
	else if(br.pier_of[c] >= 0) { v.type = 2; v.slot = clu_off[v.b] + br.pier_of[c]; }
	return v;
}

// candidate e of a type-2 cluster: chain1 + bridge + chain2
DEV bool vote_candidate2(const sgraph &sg, const vote_cluster &v, const bridge_dev &br, int e, int32_t bd0, int32_t bd3,
		int &strand, double &score, int &cn, int &wn)
{
	const int K = br.K;
	int bi = br.br_order[v.slot * 2 * K + e];
	int stride = br.p_bt[v.slot] - br.p_bs[v.slot] + 1;
	const int32_t *bc = br.chains + 2 * br.p_path_off[v.slot] + (int64_t)bi * 2 * stride;
	int bl = br.br_clen[v.slot * 2 * K + bi];
	seq3 w;
	w.p[0] = v.ch1; w.n[0] = v.n1; w.p[1] = bc; w.n[1] = bl; w.p[2] = v.ch2; w.n[2] = v.n2;
	if(!seq_increasing(w)) return false;
	strand = check_strand(sg, w);
	if(strand < 0) return false;
	cn = bl;
	score = br.br_stack[(v.slot * 2 * K + bi) * br.D];
	wn = w.size();
	if(wn >= 1 && w.at(0) <= bd0) return false;
	if(wn >= 1 && w.at(wn - 1) >= bd3) return false;
	int32_t intron = 0;
	for(int k = 0; k < wn / 2; k++) intron += w.at(2 * k + 1) - w.at(2 * k);
	int32_t length = bd3 - bd0 - intron;
	if(length < br.low) return false;
	if(length > br.high) return false;
	return true;
}

struct vote_out
{
	int32_t *type, *strand, *choices;
	double *score;
	int32_t *pick;               // index of the chosen candidate, -1 if none
	int32_t *clen, *wlen;        // lengths, then
	const int64_t *coff, *woff;  // offsets (emit pass)
	int32_t *chain, *whole;
};

KERNEL_OCC(8) k_vote(int64_t n_clu, int emit, const int32_t *c_bundle, const int64_t *clu_off, const int32_t *c_bounds, const int32_t *c_chain1,
		const int32_t *c_chain2, chains_view cv, graph_dev g, const uint8_t *b_strand, bridge_dev br, vote_out o, vote_lists vl)
{
	int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	int kind = 0;                    // 1 / 2: goes to the work list of that type
	if(c < n_clu)
	{
		const int ss = br.vp1[c], tt = br.vp2[c];
		if(!emit)
		{
			o.type[c] = -1; o.strand[c] = 0; o.choices[c] = 0; o.score[c] = 0; o.clen[c] = 0; o.wlen[c] = 0; o.pick[c] = -1;
			if(ss >= 0 && tt >= 0)
			{
				vote_cluster v = vote_load(c, ss, tt, c_bundle, clu_off, c_chain1, c_chain2, cv, br);
				if(v.type == 1 && v.n1 == 0 && v.n2 == 0)
				{
					// both mates unspliced inside overlapping vertices: `whole` is empty, only the fragment length decides
					int32_t length = c_bounds[4 * c + 3] - c_bounds[4 * c];
					if(length >= br.low && length <= br.high) { o.type[c] = 1; o.choices[c] = 1; o.score[c] = 10; o.pick[c] = 0; }
				}
				else kind = v.type;
			}
		}
		else if(o.pick[c] >= 0)
		{
			// the choice is known: rebuild its coordinates only
			vote_cluster v = vote_load(c, ss, tt, c_bundle, clu_off, c_chain1, c_chain2, cv, br);
			seq3 w, cc;
			cc.n[0] = cc.n[1] = cc.n[2] = 0; cc.p[0] = cc.p[1] = cc.p[2] = v.ch1;
			if(v.type == 1) merge_intron_chains(v.ch1, v.n1, v.ch2, v.n2, w);
			else
			{
				const int K = br.K;
				int bi = br.br_order[v.slot * 2 * K + o.pick[c]];
				int stride = br.p_bt[v.slot] - br.p_bs[v.slot] + 1;
				const int32_t *bc = br.chains + 2 * br.p_path_off[v.slot] + (int64_t)bi * 2 * stride;
				int bl = br.br_clen[v.slot * 2 * K + bi];
				w.p[0] = v.ch1; w.n[0] = v.n1; w.p[1] = bc; w.n[1] = bl; w.p[2] = v.ch2; w.n[2] = v.n2;
				cc.p[0] = bc; cc.n[0] = bl;
			}
			int nc = cc.size(), nw = w.size();
			for(int k = 0; k < nc; k++) o.chain[o.coff[c] + k] = cc.at(k);
			for(int k = 0; k < nw; k++) o.whole[o.woff[c] + k] = w.at(k);
		}
	}
	if(emit) return;
#ifndef AGPU_EMU
	const int lane = threadIdx.x & 31;
	for(int t = 1; t <= 2; t++)
	{
		const unsigned m = __ballot_sync(0xffffffffu, kind == t);
		if(!m) continue;
		int base = 0;
		if(lane == __ffs((int)m) - 1) base = atomicAdd(t == 1 ? vl.n1 : vl.n2, __popc(m));
		base = __shfl_sync(0xffffffffu, base, __ffs((int)m) - 1);
		if(kind == t) (t == 1 ? vl.list1 : vl.list2)[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)c;
	}
#else
	if(kind == 1) vl.list1[atomicAdd(vl.n1, 1)] = (int32_t)c;
	if(kind == 2) vl.list2[atomicAdd(vl.n2, 1)] = (int32_t)c;
#endif
}

KERNEL_OCC(8) k_vote_type1(int64_t n_clu, const int32_t *c_bundle, const int64_t *clu_off, const int32_t *c_bounds, const int32_t *c_chain1,
		const int32_t *c_chain2, chains_view cv, graph_dev g, const uint8_t *b_strand, bridge_dev br, vote_out o, vote_lists vl)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_clu || i >= *vl.n1) return;
	const int64_t c = vl.list1[i];
	vote_cluster v = vote_load(c, br.vp1[c], br.vp2[c], c_bundle, clu_off, c_chain1, c_chain2, cv, br);
	sgraph sg = sgraph_of(g, b_strand, v.b);
	seq3 w;
	if(!merge_intron_chains(v.ch1, v.n1, v.ch2, v.n2, w)) return;
	if(!seq_increasing(w)) return;
	int s = check_strand(sg, w);
	if(s < 0) return;
	const int32_t bd0 = c_bounds[4 * c], bd3 = c_bounds[4 * c + 3];
	int wn = w.size();
	if(wn >= 1 && w.at(0) <= bd0) return;
	if(wn >= 1 && w.at(wn - 1) >= bd3) return;
	int32_t intron = 0;
	for(int k = 0; k < wn / 2; k++) intron += w.at(2 * k + 1) - w.at(2 * k);
	int32_t length = bd3 - bd0 - intron;
	if(length < br.low || length > br.high) return;
	o.type[c] = 1; o.strand[c] = s; o.choices[c] = 1; o.score[c] = 10; o.clen[c] = 0; o.wlen[c] = wn; o.pick[c] = 0;
}

KERNEL_OCC(6) k_vote_type2(int64_t n_clu, const int32_t *c_bundle, const int64_t *clu_off, const int32_t *c_bounds, const int32_t *c_chain1,
		const int32_t *c_chain2, chains_view cv, graph_dev g, const uint8_t *b_strand, bridge_dev br, vote_out o, vote_lists vl)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_clu || i >= *vl.n2) return;
	const int64_t c = vl.list2[i];
	vote_cluster v = vote_load(c, br.vp1[c], br.vp2[c], c_bundle, clu_off, c_chain1, c_chain2, cv, br);
	sgraph sg = sgraph_of(g, b_strand, v.b);
	const int32_t bd0 = c_bounds[4 * c], bd3 = c_bounds[4 * c + 3];
	const int ncand = br.p_nbr[v.slot];
	int be = -1, choices = 0;
	for(int e = 0; e < ncand; e++)
	{
		int s = 0, cn = 0, wn = 0;
		double score = 0;
		if(!vote_candidate2(sg, v, br, e, bd0, bd3, s, score, cn, wn)) continue;
		if(be < 0) { be = e; o.type[c] = 2; o.strand[c] = s; o.score[c] = score; o.clen[c] = cn; o.wlen[c] = wn; o.pick[c] = e; }
		choices++;
	}
	if(be >= 0) o.choices[c] = choices;
}

// ---- update_bridges (rnacore/bundle_base.cc:420-507) for every bridged cluster, as looped in meta/bundle.cc:73-79
// One thread per cluster MEMBER (fragment of a frlist).  Pass 0 decides acceptance and counts; device-wide scans turn the
// per-member flags into the fcst entry order (= member order, which is cluster-major, the order of the reference's loops)
// and the offsets of the coverage stretches; pass 1 applies.
struct update_dev
{
	const int64_t *crank;        // flag rank over members: cluster of member x = crank[x + 1] - 1
	int32_t *ent_flag;           // pass 0: 0 if the member joins fcst (accepted, non-empty chain), else -1
	int32_t *gap_cnt;            // pass 0: coverage stretches (mmap += 1) of the member, 0 if not accepted
	int32_t *acc_flag;           // pass 0: 1 if accepted
	const int64_t *ent_rank;     // scanned
	const int64_t *gap_off;      // scanned
	int32_t *ent_frag, *ent_xs, *ent_len;
	int64_t *ent_voff;
	int32_t *bridged;            // [NB]
	int64_t *ex_s, *ex_e;        // the stretches as global window positions, appended after the earlier rounds' at ex_base
	int64_t ex_base;
};

KERNEL_OCC(8) k_update(int64_t n_mem, int apply, const int32_t *c_bundle, const int64_t *frg_off, const int32_t *members,
		hits_dev h, const int32_t *f_h1, const int32_t *f_h2, int32_t *f_type, const int32_t *o_type, const int32_t *o_strand,
		const int64_t *o_coff, const int32_t *o_chain, const int32_t *b_lpos, const int32_t *b_covhi, const int64_t *cov_base,
		u32 *border, update_dev u, int *err)
{
	int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(x >= n_mem) return;
	int b = -1;
	bool accepted = false;
	if(apply ? u.acc_flag[x] != 0 : true)
	{
		const int64_t c = u.crank[x + 1] - 1;
		if(o_type[c] > 0)
		{
			b = c_bundle[c];
			const int64_t f0 = frg_off[b], h0 = h.bundle_hit_off[b];
			const int32_t *chain = o_chain + o_coff[c];
			const int cl = (int)(o_coff[c + 1] - o_coff[c]);
			const int fr = members[x];
			const int64_t i1 = h0 + f_h1[f0 + fr], i2 = h0 + f_h2[f0 + fr];
			const int32_t r1 = h.rpos[i1], p2 = h.pos[i2];
			accepted = true;
			// v1 = (h1.rpos, chain..., h2.pos) must be non-decreasing when h1.rpos < h2.pos
			if(!apply && r1 < p2)
			{
				int32_t prev = r1;
				for(int k = 0; k < cl && accepted; k++) { if(prev > chain[k]) accepted = false; prev = chain[k]; }
				if(accepted && prev > p2) accepted = false;
			}
			if(accepted)
			{
				if(apply)
				{
					f_type[f0 + fr] = cl > 0 ? 2 : 1;
					if(cl > 0)
					{
						char s = '.';
						char x1 = (char)h.xs[i1], x2 = (char)h.xs[i2];
						if(x1 != '.') s = x1;
						if(x2 != '.') s = x2;
						if(x1 != '.' && x2 != '.' && x1 != x2) s = '.';
						char ss = '.';
						const int strand = o_strand[c];
						if(strand == 1) ss = '+';
						if(strand == 2) ss = '-';
						char use;
						if(s == ss) use = ss;
						else if(s != '.' && ss == '.') use = s;
						else if(ss != '.' && s == '.') use = ss;
						else use = '.';
						const int64_t eo = u.ent_rank[x];
						u.ent_frag[eo] = fr;
						u.ent_xs[eo] = use == '+' ? 1 : (use == '-' ? 2 : 0);
						u.ent_len[eo] = cl;
						u.ent_voff[eo] = o_coff[c];
					}
				}
				// mmap += 1 over every stretch (v1[2k], v1[2k+1]) with v1[2k] < v1[2k+1]: new borders + a list entry
				const int64_t cbase = cov_base[b] - (int64_t)b_lpos[b];
				int gaps = 0;
				const int nv = cl + 2;
				for(int k = 0; k < nv / 2; k++)
				{
					int32_t a = (2 * k == 0) ? r1 : chain[2 * k - 1];
					int32_t e = (2 * k + 1 == nv - 1) ? p2 : chain[2 * k];
					if(a >= e) continue;
					if(a < b_lpos[b] || e > b_covhi[b]) { if(apply) atomicAdd(&err[ERR_CAP], 1); continue; }
					if(apply)
					{
						int64_t s0 = cbase + a, e0 = cbase + e;
						int64_t at = u.ex_base + u.gap_off[x] + gaps;
						u.ex_s[at] = s0; u.ex_e[at] = e0;
						atomicOr(&border[s0 >> 5], 1u << (s0 & 31));
						atomicOr(&border[e0 >> 5], 1u << (e0 & 31));
					}
					gaps++;
				}
				if(!apply) { u.ent_flag[x] = cl > 0 ? 0 : -1; u.gap_cnt[x] = gaps; u.acc_flag[x] = 1; }
			}
		}
	}
	if(!apply)
	{
		if(!accepted) { u.ent_flag[x] = -1; u.gap_cnt[x] = 0; u.acc_flag[x] = 0; }
		return;
	}
	// bridged count of the bundle: members of a bundle are neighbours, one atomic per (warp, bundle)
#ifndef AGPU_EMU
	const unsigned act = __activemask();
	const unsigned peers = __match_any_sync(act, accepted ? b : -1);
	if(accepted && (int)(threadIdx.x & 31) == __ffs((int)peers) - 1) atomicAdd(&u.bridged[b], __popc(peers));
#else
	if(accepted) atomicAdd(&u.bridged[b], 1);
#endif
}

// fcst table insertion for the entries (elements) of all rounds so far
KERNEL k_fcst_insert(int64_t n_ent, int32_t n_bundles, const int64_t *ent_boff, const int32_t *ent_xs, const int32_t *ent_len,
		const int64_t *ent_voff, const int32_t *val, const int64_t *reg_off, u64 *slot_word, int32_t *slot_first, int32_t *slot_cnt,
		int64_t *ent_slot, int *err)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_ent) return;
	int b = find_segment(ent_boff, n_bundles, i);
	chain_src s;
	s.val = val; s.off = ent_voff; s.off32 = NULL; s.len = ent_len;
	int64_t r0 = reg_off[b];
	u32 rs = (u32)(reg_off[b + 1] - r0);
	u64 hsh = chain_hash(val + ent_voff[i], ent_len[i]);
	int64_t sl = chain_table_insert(slot_word, r0, rs, s, i, hsh);
	ent_slot[i] = sl;
	if(sl < 0) { atomicAdd(&err[ERR_CAP], 1); return; }
	atomicAdd(&slot_cnt[sl * 3 + ent_xs[i]], 1);
	atomicMin(&slot_first[sl], (int32_t)(i - ent_boff[b]));
}

// entries of bundle b after a round = entries of the earlier rounds, then the new ones
KERNEL k_merge_entries(int64_t n, int32_t n_bundles, const int64_t *m_boff, const int64_t *o_boff, const int64_t *n_boff,
		const int32_t *o_frag, const int32_t *o_xs, const int32_t *o_len, const int64_t *o_voff,
		const int32_t *n_frag, const int32_t *n_xs, const int32_t *n_len, const int64_t *n_voff, int64_t val_base,
		int32_t *m_frag, int32_t *m_xs, int32_t *m_len, int64_t *m_voff)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	int b = find_segment(m_boff, n_bundles, i);
	int64_t k = i - m_boff[b];
	int64_t no = o_boff[b + 1] - o_boff[b];
	if(k < no)
	{
		int64_t s = o_boff[b] + k;
		m_frag[i] = o_frag[s]; m_xs[i] = o_xs[s]; m_len[i] = o_len[s]; m_voff[i] = o_voff[s];
	}
	else
	{
		int64_t s = n_boff[b] + (k - no);
		m_frag[i] = n_frag[s]; m_xs[i] = n_xs[s]; m_len[i] = n_len[s]; m_voff[i] = n_voff[s] + val_base;
	}
}

KERNEL k_scatter_handle(int64_t n_ent, int32_t n_bundles, const int64_t *ent_boff, const int64_t *frg_off, const int32_t *ent_frag,
		const int32_t *ent_chain, int32_t *frag_chain)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_ent) return;
	int b = find_segment(ent_boff, n_bundles, i);
	frag_chain[frg_off[b] + ent_frag[i]] = ent_chain[i];
}

} // namespace agpu

struct bridge_state
{
	bool built = false;
	agpu::dbuf<int32_t> vp1, vp2, pier_of, n_piers, n_groups, p_bs, p_bt, p_group, g_k1, g_k2, g_first, g_last, maxin;
	agpu::dbuf<int64_t> g_rows, g_row_off, g_cand_need, g_cand_off, p_path_need, p_path_off;
	agpu::dbuf<int32_t> t_cnt, t_len, t_tr1, t_tr2, t_stack, cand, cand_idx, p_nbr, br_len, br_clen, br_stack, br_order, paths, chains;
	agpu::dbuf<agpu::u64> key_scratch;
	// opt
	agpu::dbuf<int32_t> o_type, o_strand, o_choices, o_clen, o_wlen, o_chain, o_whole;
	agpu::dbuf<double> o_score;
	agpu::dbuf<int64_t> o_coff, o_woff;
	int64_t n_clu = 0, n_cval = 0, n_wval = 0;
	bool updated = false;
};

// update / fcst entries of all update rounds: a re-bridge (group pass) starts a new bridge_state and appends to these
struct bridge_entries
{
	agpu::dbuf<int32_t> ent_frag, ent_xs, ent_len, fc_val, frag_chain;
	agpu::dbuf<int64_t> ent_voff, ent_boff;
	int64_t n_ent = 0, n_chain_val = 0;
};

#endif
