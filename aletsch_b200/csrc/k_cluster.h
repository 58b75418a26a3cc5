// Stage 3b kernels: paired-read clustering (rnacore/graph_cluster.cc).
//
//   group_pereads            :28-91    align both mates of every to-be-bridged fragment to vertex paths and
//                                      group fragments by the pair of paths, groups in first-seen order
//   align_hit_to_splice_graph rnacore/essential.cc:461-472 -> build_path_from_mixed_coordinates :405-434
//                             -> build_path_from_intron_coordinates :368-403, check_continuous_vertices :436-446
//   build_pereads_clusters   :93-168   per group 4-level gap partition, bounds = first + sum(x - first) / count
//   partition                :170-203  std::sort per level (unstable: the libstdc++ permutation is reproduced)
//
// A vertex path is compared in run-length form (maximal runs of consecutive vertex numbers): the runs
// of a spliced mate are the runs of its intron chain's path (computed once per chain) with the first run
// stretched down to the vertex holding pos and the last run stretched up to the vertex holding rpos - 1.
#ifndef ALETSCH_B200_CSRC_K_CLUSTER_H
#define ALETSCH_B200_CSRC_K_CLUSTER_H

#include "runtime.h"
#include "k_graph.h"
#include "stdsort.h"

namespace agpu {

struct gview                     // read-only view of the graph of one bundle
{
	int nv;
	const int32_t *v_l, *v_r, *v_brk;
};

DEV gview graph_of(const graph_dev &g, int b)
{
	gview v;
	b = graph_index(g, b);
	int64_t v0 = vert_base(g, b);
	v.nv = g.n_pex[b] + 2;
	v.v_l = g.v_l + v0; v.v_r = g.v_r + v0; v.v_brk = g.v_brk + v0;
	return v;
}

// splice_graph::locate_vertex(p) (rnacore/splice_graph.cc:1166-1215)
DEV int locate_vertex(const gview &g, int32_t p)
{
	int a = 1, b = g.nv - 1;
	int m = -1;
	while(a < b)
	{
		int mid = (a + b) / 2;
		if(p >= g.v_l[mid] && p < g.v_r[mid]) { m = mid; break; }
		if(p < g.v_l[mid]) b = mid;
		else a = mid + 1;
	}
	if(m < 0) m = b;
	if(p >= g.v_l[m] && p < g.v_r[m]) return m;
	return -1;
}

// rindex[p] (vertices 0 .. n-1 keyed by rpos) and lindex[q] (vertices 1 .. n keyed by lpos); -1 if absent
DEV int rindex_find(const gview &g, int32_t p)
{
	int k = lower_bound_idx(g.v_r, g.nv - 1, p);
	return (k < g.nv - 1 && g.v_r[k] == p) ? k : -1;
}
DEV int lindex_find(const gview &g, int32_t q)
{
	int k = lower_bound_idx(g.v_l + 1, g.nv - 1, q) + 1;
	return (k < g.nv && g.v_l[k] == q) ? k : -1;
}
// check_continuous_vertices(x, y)
DEV bool continuous(const gview &g, int x, int y) { return x >= y || (g.v_brk[y] - g.v_brk[x]) == 0; }

// per chain record: path of the intron chain in the bundle's graph, in run-length form
struct chain_paths
{
	int32_t *valid;          // build_path_from_intron_coordinates succeeded
	int32_t *mono;           // chain coordinates non-decreasing
	int32_t *first, *last;   // chain.front(), chain.back()
	int32_t *nruns;
	int32_t *runs;           // pairs (start, end) at run_base(record)
};

// run storage of the chain record at scratch slot e (its representative element's coordinates start at voff):
// records own disjoint windows of len + 2 ints
HD int64_t run_base(int64_t rep_elem, int64_t voff) { return voff + 2 * rep_elem; }

KERNEL k_chain_paths(int64_t n_elem, const int32_t *elem_bundle, chains_view cv, graph_dev g, chain_paths cp)
{
	int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(e >= n_elem) return;
	int b = elem_bundle[e];
	int k = (int)(e - cv.elem_off[b]);
	if(k >= cv.n_chains[b]) return;
	if(graph_index(g, b) < 0) return;             // bundle outside every cluster of bundles (group pass only)
	gview gv = graph_of(g, b);
	int len = cv.len(b, k);
	const int32_t *v = cv.ptr(b, k);
	int64_t rep = cv.elem_off[b] + cv.c_rep[cv.elem_off[b] + k];
	int64_t voff = cv.voff64 ? cv.voff64[rep] : (int64_t)cv.voff32[rep];
	int32_t *runs = cp.runs + run_base(rep, voff);
	bool mono = true;
	for(int i = 0; i + 1 < len; i++) if(v[i] > v[i + 1]) mono = false;
	cp.mono[e] = mono ? 1 : 0;
	cp.first[e] = len > 0 ? v[0] : 0;
	cp.last[e] = len > 0 ? v[len - 1] : 0;
	int n = len / 2;
	bool ok = (len > 0 && (len & 1) == 0);
	int nr = 0;
	int prev_kq = -1;
	for(int i = 0; ok && i < n; i++)
	{
		int32_t p = v[2 * i], q = v[2 * i + 1];
		if(p >= q) { ok = false; break; }
		int kp = rindex_find(gv, p), kq = lindex_find(gv, q);
		if(kp < 0 || kq < 0) { ok = false; break; }
		if(i == 0) { runs[0] = kp; runs[1] = kp; nr = 1; }
		else
		{
			// vertices prev_kq .. kp must be continuous
			if(prev_kq > kp || !continuous(gv, prev_kq, kp)) { ok = false; break; }
			// append range prev_kq .. kp to the run list
			if(runs[2 * nr - 1] + 1 == prev_kq) runs[2 * nr - 1] = kp;
			else { runs[2 * nr] = prev_kq; runs[2 * nr + 1] = kp; nr++; }
		}
		prev_kq = kq;
	}
	if(ok)
	{
		// the path ends with pp.back().second
		if(runs[2 * nr - 1] + 1 == prev_kq) runs[2 * nr - 1] = prev_kq;
		else { runs[2 * nr] = prev_kq; runs[2 * nr + 1] = prev_kq; nr++; }
	}
	cp.valid[e] = ok ? 1 : 0;
	cp.nruns[e] = ok ? nr : 0;
}

// aligned mate: runs of its vertex path are (a1 .. runs[0].end), runs[1..nr-2], (runs[nr-1].start .. a2)
struct mate_path
{
	int32_t a1, a2;          // first / last vertex of the path
	int32_t nr;              // number of runs (1 if the mate has no chain)
	const int32_t *runs;     // chain runs (NULL without chain)
	DEV int32_t rs(int i) const { int32_t s = runs ? runs[2 * i] : a1; return i == 0 ? a1 : s; }
	DEV int32_t re(int i) const { int32_t e = runs ? runs[2 * i + 1] : a2; return i == nr - 1 ? a2 : e; }
};

struct cluster_dev
{
	// per fragment (global index)
	int32_t *f_ok;                       // both mates aligned
	int32_t *m_a1, *m_a2;                // [2F] per mate
	u64 *f_hash;
	int64_t *f_slot;
	int32_t *f_next;                     // arrival rank of the fragment inside its group (0 .. slot_n - 1, any order)
	// group table
	const int64_t *reg_off;
	u64 *slot_word;
	int32_t *slot_min, *slot_n, *slot_head;
};

DEV mate_path mate_of(const chains_view &cv, const chain_paths &cp, const cluster_dev &c, const int32_t *handle_chain,
		int b, int64_t hit, int64_t f, int which)
{
	mate_path m;
	m.a1 = c.m_a1[2 * f + which]; m.a2 = c.m_a2[2 * f + which];
	int ch = handle_chain[hit];
	if(ch < 0) { m.nr = 1; m.runs = NULL; return m; }
	int64_t e = cv.elem_off[b] + ch;
	int64_t rep = cv.elem_off[b] + cv.c_rep[e];
	int64_t voff = cv.voff64 ? cv.voff64[rep] : (int64_t)cv.voff32[rep];
	m.nr = cp.nruns[e];
	m.runs = cp.runs + run_base(rep, voff);
	return m;
}

DEV bool same_path(const mate_path &x, const mate_path &y)
{
	if(x.nr != y.nr) return false;
	for(int i = 0; i < x.nr; i++) if(x.rs(i) != y.rs(i) || x.re(i) != y.re(i)) return false;
	return true;
}

DEV u64 path_hash(const mate_path &x, u64 h)
{
	h = mix64(h ^ (u64)x.nr);
	for(int i = 0; i < x.nr; i++) h = mix64(h ^ (((u64)(u32)x.rs(i) << 32) | (u64)(u32)x.re(i)));
	return h;
}

// ---- C1: align both mates of every to-be-bridged fragment; frgs[i][2] := -1, then 0 if both align
KERNEL_OCC(8) k_frag_align(int64_t n_frg, const int32_t *f_bundle, const int64_t *frg_off, hits_dev h, const int32_t *f_h1, const int32_t *f_h2,
		int32_t *f_type, chains_view cv, chain_paths cp, const int32_t *handle_chain, graph_dev g, cluster_dev c)
{
	int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(f >= n_frg) return;
	c.f_ok[f] = 0;
	c.f_slot[f] = -1;
	int b = f_bundle[f];
	if(graph_index(g, b) < 0) return;             // bundle outside every cluster of bundles (group pass only)
	if(f_type[f] != 0) return;                    // only unbridged fragments are grouped (:37-38)
	f_type[f] = -1;
	int64_t h0 = h.bundle_hit_off[b];
	int64_t i1 = h0 + f_h1[f], i2 = h0 + f_h2[f];
	if(h.pos[i1] > h.pos[i2]) return;
	if(h.rpos[i1] > h.rpos[i2]) return;
	gview gv = graph_of(g, b);
	u64 hsh = 0x1234567ULL;
	for(int w = 0; w < 2; w++)
	{
		int64_t hi = w == 0 ? i1 : i2;
		int32_t pos = h.pos[hi], rpos = h.rpos[hi];
		int ch = handle_chain[hi];
		int64_t e = ch >= 0 ? cv.elem_off[b] + ch : -1;
		// check_increasing_sequence(pos, chain..., rpos)
		if(ch >= 0) { if(!cp.mono[e] || pos > cp.first[e] || cp.last[e] > rpos) return; }
		else if(pos > rpos) return;
		int u1 = locate_vertex(gv, pos), u2 = locate_vertex(gv, rpos - 1);
		if(u1 < 0 || u2 < 0) return;
		if(u1 > u2) return;
		int32_t a1 = u1, a2 = u2;
		if(ch >= 0)
		{
			if(!cp.valid[e]) return;
			int64_t rep = cv.elem_off[b] + cv.c_rep[e];
			int64_t voff = cv.voff64 ? cv.voff64[rep] : (int64_t)cv.voff32[rep];
			const int32_t *runs = cp.runs + run_base(rep, voff);
			int nr = cp.nruns[e];
			int32_t front = runs[0], back = runs[2 * nr - 1];
			if(front < a1) a1 = front;             // for(i = u1; i < uu.front(); i++) adds nothing when u1 >= uu.front()
			if(back > a2) a2 = back;
		}
		c.m_a1[2 * f + w] = a1; c.m_a2[2 * f + w] = a2;
	}
	f_type[f] = 0;
	c.f_ok[f] = 1;
	mate_path p1 = mate_of(cv, cp, c, handle_chain, b, i1, f, 0), p2 = mate_of(cv, cp, c, handle_chain, b, i2, f, 1);
	hsh = path_hash(p2, path_hash(p1, hsh));
	c.f_hash[f] = hsh;
}

// ---- C2: group by (path1, path2): per-bundle table, exact comparison against the slot's first claimer
KERNEL_OCC(8) k_frag_group(int64_t n_frg, const int32_t *f_bundle, const int64_t *frg_off, hits_dev h, const int32_t *f_h1, const int32_t *f_h2,
		chains_view cv, chain_paths cp, const int32_t *handle_chain, cluster_dev c, int *err)
{
	int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(f >= n_frg) return;
	if(!c.f_ok[f]) return;
	int b = f_bundle[f];
	int64_t h0 = h.bundle_hit_off[b];
	int64_t r0 = c.reg_off[b];
	u32 mask = (u32)(c.reg_off[b + 1] - r0) - 1;
	u64 hsh = c.f_hash[f];
	u32 pos = (u32)(hsh >> 7) & mask;
	u64 mine = ((hsh >> 32) << 32) | (u64)(u32)(f + 1);
	mate_path p1 = mate_of(cv, cp, c, handle_chain, b, h0 + f_h1[f], f, 0), p2 = mate_of(cv, cp, c, handle_chain, b, h0 + f_h2[f], f, 1);
	int64_t sl = -1;
	for(u32 probe = 0; probe <= mask; probe++)
	{
		u64 cur = atomicCAS(&c.slot_word[r0 + pos], (u64)0, mine);
		if(cur == 0) { sl = r0 + pos; break; }
		if((cur >> 32) == (mine >> 32))
		{
			int64_t rf = (int64_t)(u32)(cur & 0xffffffffULL) - 1;
			mate_path q1 = mate_of(cv, cp, c, handle_chain, b, h0 + f_h1[rf], rf, 0), q2 = mate_of(cv, cp, c, handle_chain, b, h0 + f_h2[rf], rf, 1);
			if(same_path(p1, q1) && same_path(p2, q2)) { sl = r0 + pos; break; }
		}
		pos = (pos + 1) & mask;
	}
	if(sl < 0) { atomicAdd(&err[ERR_CAP], 1); c.f_ok[f] = 0; return; }
	c.f_slot[f] = sl;
	int32_t lf = (int32_t)(f - frg_off[b]);
	atomicMin(&c.slot_min[sl], lf);
	c.f_next[f] = atomicAdd(&c.slot_n[sl], 1);
}

// members of every group side by side (unordered inside the group): fragment f goes to its group's window at its arrival rank
KERNEL k_members_scatter(int64_t n_frg, const int32_t *f_bundle, const int64_t *frg_off, cluster_dev c, const int64_t *member_off, int32_t *members)
{
	int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(f >= n_frg) return;
	int64_t sl = c.f_slot[f];
	if(sl < 0) return;
	int64_t f0 = frg_off[f_bundle[f]];
	members[member_off[f0 + c.slot_min[sl]] + c.f_next[f]] = (int32_t)(f - f0);
}

// leader[f] = group size if f is the first fragment of its group, else -1 (input of the flag scans)
#define BIG_GROUP 16            // groups up to this size: one thread, insertion sorts only (std::sort on <= 16 elements); above: a whole
                                // warp (CUDA build).  One thread replaying introsort in local memory for 17 .. 48 members was measured 2x slower.
#define LANE_RANGE 16           // inside the warp kernel, ranges up to this size are sorted by a single lane
#define WARP_EL_CAP 128         // groups up to this size are partitioned in shared memory (4 warps x 1 KB per CTA)

// small_list / big_list: the leaders packed densely (any order), so that the partition kernels run with full warps
KERNEL k_group_leaders(int64_t n_frg, const int32_t *f_bundle, const int64_t *frg_off, cluster_dev c, int32_t *leader, int32_t *leader_size,
		int32_t *n_big, int32_t *big_list, int32_t big_cap, int32_t *n_small, int32_t *small_list)
{
	int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	bool lead = false;
	int size = 0;
	if(f < n_frg)
	{
		leader[f] = -1;
		leader_size[f] = 0;
		int64_t sl = c.f_slot[f];
		if(sl >= 0)
		{
			int b = f_bundle[f];
			if(c.slot_min[sl] == (int32_t)(f - frg_off[b]))
			{
				lead = true;
				size = c.slot_n[sl];
				leader[f] = 1;
				leader_size[f] = size;
			}
		}
	}
#ifndef AGPU_EMU
	if(lead && size > BIG_GROUP)
	{
		int k = atomicAdd(n_big, 1);
		if(k < big_cap) big_list[k] = (int32_t)f;
		atomicAdd(n_big + 1, size);              // members the warp kernel handles (agpu_counts::big_group_members)
	}
	// one atomic per warp for the small groups
	const bool small = lead && size <= BIG_GROUP;
	const unsigned m = __ballot_sync(0xffffffffu, small);
	if(m)
	{
		const int lane = threadIdx.x & 31;
		int base = 0;
		if(lane == __ffs((int)m) - 1) base = atomicAdd(n_small, __popc(m));
		base = __shfl_sync(0xffffffffu, base, __ffs((int)m) - 1);
		if(small) small_list[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)f;
	}
#else
	if(lead) small_list[atomicAdd(n_small, 1)] = (int32_t)f;
	(void)n_big; (void)big_list; (void)big_cap;
#endif
}

struct part_ctx
{
	u64 *el;                     // elements of the group: key of the current level in the high word, fragment in the low word
	int32_t *cflag;              // cluster-start flags parallel to el
	const int32_t *f_h1, *f_h2;  // bundle's fragments
	const int32_t *pos, *rpos;   // bundle's hits
	int gap;
	HD int32_t key(int r, int32_t fr) const
	{
		int32_t hh = (r < 2) ? f_h1[fr] : f_h2[fr];
		return (r & 1) ? rpos[hh] : pos[hh];
	}
};

// compare_rank0..3 (rnacore/graph_cluster.cc:205-208) on elements that carry their key in the high word
// (biased so that the unsigned order of the word is the signed order of the key)
struct key_less
{
	HD bool operator()(u64 x, u64 y) const { return (x >> 32) < (y >> 32); }
};
HD u64 pack_key(int32_t key, int32_t fr) { return ((u64)((u32)key ^ 0x80000000u) << 32) | (u64)(u32)fr; }
HD int32_t unpack_key(u64 e) { return (int32_t)((u32)(e >> 32) ^ 0x80000000u); }

// graph_cluster::partition (rnacore/graph_cluster.cc:170-203), in place on the member array
template<int R> DEV void partition_rec(const part_ctx &c, int lo, int hi)
{
	for(int k = lo; k < hi; k++) { int32_t fr = (int32_t)(u32)(c.el[k] & 0xffffffffULL); c.el[k] = pack_key(c.key(R, fr), fr); }
	key_less less;
	std_sort_handles(c.el + lo, hi - lo, less);
	int pre = lo;
	for(int k = lo + 1; k <= hi; k++)
	{
		if(k < hi && unpack_key(c.el[k]) - unpack_key(c.el[k - 1]) <= c.gap) continue;
		partition_rec<R + 1>(c, pre, k);
		pre = k;
	}
}
template<> DEV void partition_rec<4>(const part_ctx &c, int lo, int hi) { (void)hi; c.cflag[lo] = 1; }

// ---- C3: the first fragment of every group gathers the members (ascending fragment index) and partitions them
KERNEL k_group_partition(int64_t n_frg, const int32_t *f_bundle, const int64_t *frg_off, hits_dev h, const int32_t *f_h1, const int32_t *f_h2,
		cluster_dev c, const int32_t *n_small, const int32_t *small_list, const int64_t *member_off, int32_t *members, u64 *elems,
		int32_t *cflag, int gap)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_frg || i >= *n_small) return;
	const int64_t f = small_list[i];                 // groups above BIG_GROUP members are handled by k_group_partition_warp
	int b = f_bundle[f];
	int64_t f0 = frg_off[b];
	int64_t sl = c.f_slot[f];
	int n = c.slot_n[sl];
	int32_t *m = members + member_off[f];
#ifndef AGPU_EMU
	{
		// at most 16 members: everything stays in thread-local memory, and std::sort on <= 16 elements is a stable
		// insertion sort (__final_insertion_sort -> __insertion_sort)
		const int32_t *fh1 = f_h1 + f0, *fh2 = f_h2 + f0;
		const int32_t *hp = h.pos + h.bundle_hit_off[b], *hr = h.rpos + h.bundle_hit_off[b];
		u64 e[BIG_GROUP];
		for(int k = 0; k < n; k++) e[k] = (u64)(u32)m[k];
		for(int a = 1; a < n; a++)              // ascending fragment index
		{
			u64 v = e[a];
			int q = a - 1;
			while(q >= 0 && e[q] > v) { e[q + 1] = e[q]; q--; }
			e[q + 1] = v;
		}
		unsigned starts = 1u;
		for(int r = 0; r < 4; r++)
		{
			for(int i = 0; i < n; i++)
			{
				int32_t fr = (int32_t)(u32)(e[i] & 0xffffffffULL);
				int32_t hh = (r < 2) ? fh1[fr] : fh2[fr];
				e[i] = pack_key((r & 1) ? hr[hh] : hp[hh], fr);
			}
			for(int i = 1; i < n; i++)
			{
				if((starts >> i) & 1u) continue;          // first element of a range
				u64 v = e[i];
				int q = i - 1;
				while((v >> 32) < (e[q] >> 32)) { e[q + 1] = e[q]; q--; if((starts >> (q + 1)) & 1u) break; }
				e[q + 1] = v;
			}
			for(int i = 1; i < n; i++)
				if(!((starts >> i) & 1u) && unpack_key(e[i]) - unpack_key(e[i - 1]) > gap) starts |= 1u << i;
		}
		int32_t *cf = cflag + member_off[f];
		for(int i = 0; i < n; i++) { m[i] = (int32_t)(u32)(e[i] & 0xffffffffULL); cf[i] = (starts >> i) & 1u; }
		return;
	}
#else
	// ascending fragment index = the order group_pereads appended them (heap sort, keys are distinct)
	for(int i = n / 2 - 1; i >= 0; i--)
	{
		int root = i;
		while(true)
		{
			int ch = 2 * root + 1;
			if(ch >= n) break;
			if(ch + 1 < n && m[ch + 1] > m[ch]) ch++;
			if(m[root] >= m[ch]) break;
			int32_t t = m[root]; m[root] = m[ch]; m[ch] = t;
			root = ch;
		}
	}
	for(int end = n - 1; end > 0; end--)
	{
		int32_t t = m[0]; m[0] = m[end]; m[end] = t;
		int root = 0;
		while(true)
		{
			int ch = 2 * root + 1;
			if(ch >= end) break;
			if(ch + 1 < end && m[ch + 1] > m[ch]) ch++;
			if(m[root] >= m[ch]) break;
			int32_t t2 = m[root]; m[root] = m[ch]; m[ch] = t2;
			root = ch;
		}
	}
	part_ctx pc;
	pc.el = elems + member_off[f]; pc.cflag = cflag + member_off[f];
	for(int i = 0; i < n; i++) pc.el[i] = (u64)(u32)m[i];
	pc.f_h1 = f_h1 + f0; pc.f_h2 = f_h2 + f0;
	pc.pos = h.pos + h.bundle_hit_off[b]; pc.rpos = h.rpos + h.bundle_hit_off[b];
	pc.gap = gap;
	partition_rec<0>(pc, 0, n);
	for(int i = 0; i < n; i++) m[i] = (int32_t)(u32)(pc.el[i] & 0xffffffffULL);
#endif
}

#ifndef AGPU_EMU
// The introsort loop of std::sort (libstdc++: __introsort_loop, see stdsort.h) for 17 .. 32 elements held ONE PER LANE, lanes
// [f0, l0): the median-of-three, the partition step (the k-th element from the left that is not less than the pivot swaps with
// the k-th from the right that the pivot is not less than, while the former lies left of the latter) and the cut are bit
// arithmetic on two ballots (__fns finds the k-th set bit), the swaps one shuffle.  On return every lane of the range knows the
// leaf (first lane, length <= 16) whose stable insertion sort finishes std::sort; the caller ranks the elements inside the leaves.
// The depth-limit fallback (heap sort) goes through shared memory `sh`, sequentially, like the reference's.
__device__ __forceinline__ u32 ws32_key(u64 e) { return (u32)(e >> 32); }
__device__ void warp_sort32_loop(u64 &x, int f0, int l0, int lane, int &leaf_f, int &leaf_len, u64 *sh)
{
	const unsigned FULL = 0xffffffffu;
	const unsigned below = (1u << lane) - 1u, above = lane == 31 ? 0u : (0xffffffffu << (lane + 1));
	const int n = l0 - f0;
	int lg = 0;
	while((n >> (lg + 1)) != 0) lg++;
	int st_f[24], st_l[24], st_d[24];
	int sp = 1;
	st_f[0] = f0; st_l[0] = l0; st_d[0] = lg * 2;
	while(sp > 0)
	{
		--sp;
		int f = st_f[sp], l = st_l[sp], d = st_d[sp];
		while(l - f > 16)
		{
			if(d == 0)
			{
				sh[lane] = x;
				__syncwarp();
				if(lane == 0) { key_less less; std_sort_emul<u64, key_less> seq(sh, less); seq.partial_sort_all(f, l); }
				__syncwarp();
				x = sh[lane];
				__syncwarp();
				if(lane >= f && lane < l) { leaf_f = lane; leaf_len = 1; }
				f = l;
				break;
			}
			--d;
			const int mid = f + (l - f) / 2;
			const u32 kx = ws32_key(__shfl_sync(FULL, x, f + 1)), ky = ws32_key(__shfl_sync(FULL, x, mid)), kz = ws32_key(__shfl_sync(FULL, x, l - 1));
			int p;                                                        // __move_median_to_first(f, f + 1, mid, l - 1)
			if(kx < ky) { if(ky < kz) p = mid; else if(kx < kz) p = l - 1; else p = f + 1; }
			else if(kx < kz) p = f + 1;
			else if(ky < kz) p = l - 1;
			else p = mid;
			{
				const u64 vf = __shfl_sync(FULL, x, f), vp = __shfl_sync(FULL, x, p);
				if(lane == f) x = vp; else if(lane == p) x = vf;
			}
			const u32 kp = ws32_key(__shfl_sync(FULL, x, f)), kme = ws32_key(x);
			const bool valid = lane > f && lane < l;
			const bool ge = valid && !(kme < kp), le = valid && !(kp < kme);
			const unsigned mg = __ballot_sync(FULL, ge), ml = __ballot_sync(FULL, le);
			const int nL = __popc(mg), nR = __popc(ml);
			int src = lane;
			bool left = false;
			if(ge)
			{
				const int k = __popc(mg & below);
				if(k < nR) { const unsigned y = __fns(ml, 31, -(k + 1)); if((unsigned)lane < y) { src = (int)y; left = true; } }
			}
			const int K = __popc(__ballot_sync(FULL, left));
			if(le && !left)
			{
				const int k2 = __popc(ml & above);
				if(k2 < nL) { const unsigned z = __fns(mg, 0, k2 + 1); if(z < (unsigned)lane) src = (int)z; }
			}
			x = __shfl_sync(FULL, x, src);
			int cut = l;
			if(K > 0) cut = (int)__fns(ml, 31, -K);
			if(K < nL) { const int lk = (int)__fns(mg, 0, K + 1); if(lk < cut) cut = lk; }
			st_f[sp] = cut; st_l[sp] = l; st_d[sp] = d; sp++;
			l = cut;
		}
		if(l - f > 0 && lane >= f && lane < l) { leaf_f = f; leaf_len = l - f; }
	}
}

// One level of graph_cluster::partition for a group of <= 32 elements, one per lane: std::sort of every current range (range
// starts = lanes with sf set) by the key in the high word.
__device__ void warp_sort_level32(u64 &x, bool have, bool sf, int n, int lane, u64 *sh)
{
	const unsigned FULL = 0xffffffffu;
	const unsigned ms = __ballot_sync(FULL, have && sf);     // range starts; bit 0 is always set
	const int lo = 31 - __clz(ms & (0xffffffffu >> (31 - lane)));
	const unsigned up = lane == 31 ? 0u : (ms & (0xffffffffu << (lane + 1)));
	const int hi = up ? __ffs((int)up) - 1 : n;
	int leaf_f = have ? lo : lane, leaf_len = have ? hi - lo : 0;
	// at most one range of a group of <= 32 exceeds 16 elements: the introsort loop runs on that one
	const unsigned big = __ballot_sync(FULL, have && sf && hi - lo > 16);
	if(big)
	{
		const int s0 = __ffs((int)big) - 1, e0 = __shfl_sync(FULL, hi, s0);
		warp_sort32_loop(x, s0, e0, lane, leaf_f, leaf_len, sh);
	}
	// every element ranks itself inside its leaf: the stable order the insertion sorts of std::sort leave
	int rk = 0;
	const u32 kv = (u32)(x >> 32);
	for(int j = 0; j < 16; j++)
	{
		const int idx = leaf_f + j;
		const u64 o = __shfl_sync(FULL, x, idx & 31);
		if(j < leaf_len) { const u32 ko = (u32)(o >> 32); rk += (ko < kv || (ko == kv && idx < lane)) ? 1 : 0; }
	}
	if(have) sh[leaf_f + rk] = x;
	__syncwarp();
	if(have) x = sh[lane];
	__syncwarp();
}

// The same for a group of up to WARP_EL_CAP elements in shared memory (range starts = sf[i] set): the introsort loop on the
// ranges above 16 elements (whole warp, one range after the other), then ONE pass in which every element ranks itself inside
// its leaf.  srl: WARP_EL_CAP ints (range list), sscr: 2 * WARP_EL_CAP ints, sseg: WARP_EL_CAP ints.
__device__ void warp_sort_level128(u64 *el, int n, const unsigned char *sf, int *srl, int *sscr, int *sseg, int lane)
{
	const unsigned FULL = 0xffffffffu;
	key_less less;
	int nr = 0;
	for(int base = 0; base < n; base += 32)
	{
		int i = base + lane;
		bool st = i < n && sf[i];
		unsigned m = __ballot_sync(FULL, st);
		if(st) srl[nr + __popc(m & ((1u << lane) - 1u))] = i;
		nr += __popc(m);
	}
	__syncwarp();
	for(int k = 0; k < nr; k++)
	{
		int lo = srl[k], hi = (k + 1 < nr) ? srl[k + 1] : n;
		if(hi - lo > LANE_RANGE) warp_std_sort_loop(el + lo, hi - lo, less, sscr, sseg + lo, lo);
		else if(lane < hi - lo) sseg[lo + lane] = (lo << 8) | (hi - lo);
	}
	__syncwarp();
	u64 v[WARP_EL_CAP / 32];
	int dst[WARP_EL_CAP / 32];
#pragma unroll
	for(int q = 0; q < WARP_EL_CAP / 32; q++)
	{
		const int i = lane + 32 * q;
		dst[q] = -1;
		if(i < n)
		{
			v[q] = el[i];
			const int s = sseg[i], f = s >> 8, len = s & 0xff;
			const u32 kv = (u32)(v[q] >> 32);
			int rk = 0;
			for(int j = f; j < f + len; j++)
			{
				const u32 kw = (u32)(el[j] >> 32);
				rk += (kw < kv || (kw == kv && j < i)) ? 1 : 0;
			}
			dst[q] = f + rk;
		}
	}
	__syncwarp();
#pragma unroll
	for(int q = 0; q < WARP_EL_CAP / 32; q++) if(dst[q] >= 0) el[dst[q]] = v[q];
	__syncwarp();
}

// One warp per big group: members gathered in fragment order by scanning the bundle's fragments, then the four
// partition levels breadth first.  A level = (re)key every element, sort every current range with the std::sort
// permutation (big ranges by the whole warp, small ones one lane each), then open a new range wherever the gap
// between neighbours exceeds max_reads_partition_gap.  Range starts are flags by position, so the clusters come
// out in the same left-to-right order as the reference's recursion.
__global__ void k_group_partition_warp(const int32_t *n_big, const int32_t *big_list, int32_t big_cap, const int32_t *f_bundle, const int64_t *frg_off,
		hits_dev h, const int32_t *f_h1, const int32_t *f_h2, cluster_dev c, const int64_t *member_off, int32_t *members, u64 *elems,
		int32_t *cflag, int32_t *scratch, int gap)
{
	// the element array of a group of up to WARP_EL_CAP members lives in shared memory while its four levels are sorted:
	// the per-lane std::sort replays are chains of dependent element reads and moves
	__shared__ u64 s_el[4][WARP_EL_CAP];
	__shared__ int s_tmp[4][4 * WARP_EL_CAP];        // range list, two position lists of the partition steps, leaf of every element
	__shared__ unsigned char s_flag[4][WARP_EL_CAP];
	const unsigned FULL = 0xffffffffu;
	const int lane = threadIdx.x & 31;
	int nb_ = *n_big;
	if(nb_ > big_cap) nb_ = big_cap;
	const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
	for(int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < nb_; w += n_warps)
	{
	const int64_t f = big_list[w];
	const int b = f_bundle[f];
	const int64_t f0 = frg_off[b];
	const int nfb = (int)(frg_off[b + 1] - f0);
	const int64_t sl = c.f_slot[f];
	const int n = c.slot_n[sl];
	const int64_t mo = member_off[f];
	u64 *el = n <= WARP_EL_CAP ? s_el[(threadIdx.x >> 5) & 3] : elems + mo;
	int32_t *flag = cflag + mo;
	int32_t *rl = scratch + 4 * mo;              // range list (n ints), then 3n ints of sort scratch
	int32_t *ss = rl + n;
	part_ctx pc;
	pc.el = el; pc.cflag = flag;
	pc.f_h1 = f_h1 + f0; pc.f_h2 = f_h2 + f0;
	pc.pos = h.pos + h.bundle_hit_off[b]; pc.rpos = h.rpos + h.bundle_hit_off[b];
	pc.gap = gap;
	if(n <= 32)
	{
		// ---- 17 .. 32 members (nine in ten of the big groups at configs[1]): one element per lane, the four levels in registers
		u64 *sh = s_el[(threadIdx.x >> 5) & 3];
		const bool have = lane < n;
		u64 x = have ? (u64)(u32)members[mo + lane] : ~0ULL;          // the group's window, unordered
		{
			int rk = 0;                                              // ascending fragment index: rank by counting (distinct values)
			for(int j = 0; j < n; j++) { const u64 o = __shfl_sync(FULL, x, j); rk += o < x ? 1 : 0; }
			if(have) sh[rk] = x;
			__syncwarp();
			if(have) x = sh[lane];
			__syncwarp();
		}
		// the four keys of every fragment are loaded ONCE (two rounds of dependent loads instead of eight) and stay in the lane
		// that loaded them; the element that travels through the sorts carries that lane's number in its low word (the
		// comparisons only read the key in the high word), and a level fetches its key with one shuffle
		const int32_t fr0 = (int32_t)(u32)(x & 0xffffffffULL);
		int32_t k0 = 0, k1 = 0, k2 = 0, k3 = 0;
		if(have)
		{
			const int32_t h1 = pc.f_h1[fr0], h2 = pc.f_h2[fr0];
			k0 = pc.pos[h1]; k1 = pc.rpos[h1]; k2 = pc.pos[h2]; k3 = pc.rpos[h2];
		}
		x = (u64)(u32)lane;
		bool sf = lane == 0;
		for(int r = 0; r < 4; r++)
		{
			const int slot = (int)(x & 31u);
			const int32_t kr = __shfl_sync(FULL, r == 0 ? k0 : (r == 1 ? k1 : (r == 2 ? k2 : k3)), slot);
			if(have) x = pack_key(kr, slot);
			warp_sort_level32(x, have, sf, n, lane, sh);
			const u64 prev = __shfl_up_sync(FULL, x, 1);
			if(have && lane > 0 && !sf && unpack_key(x) - unpack_key(prev) > gap) sf = true;
		}
		const int32_t fr_out = __shfl_sync(FULL, fr0, (int)(x & 31u));
		if(have) { members[mo + lane] = fr_out; flag[lane] = sf ? 1 : 0; }
		__syncwarp();
		continue;
	}
	// members in ascending fragment index
	if(n <= 1024 && (int64_t)n * n < (int64_t)nfb * 4)
	{
		// moderate group inside a big bundle (n^2 / 32 steps beat the nfb / 32 steps of the scan below): order the scattered
	// window by counting smaller members
		u64 *tmp = (u64*)rl;                 // 4n ints of scratch are free at this point (8-byte aligned: 4 * mo ints)
		for(int i = lane; i < n; i += 32) tmp[i] = (u64)(u32)members[mo + i];      // the group's window, unordered
		__syncwarp();
		for(int i = lane; i < n; i += 32)
		{
			u64 v = tmp[i];
			int rk = 0;
			for(int j = 0; j < n; j++) rk += tmp[j] < v;
			el[rk] = v;
		}
	}
	else
	{
		int cnt = 0;
		for(int base = 0; base < nfb; base += 32)
		{
			int i = base + lane;
			bool in = i < nfb && c.f_slot[f0 + i] == sl;
			unsigned m = __ballot_sync(FULL, in);
			if(in) el[cnt + __popc(m & ((1u << lane) - 1u))] = (u64)(u32)i;
			cnt += __popc(m);
		}
	}
	__syncwarp();
	key_less less;
	if(n <= WARP_EL_CAP)
	{
		// everything of the group in shared memory.  A level: re-key, list the ranges, run the introsort loop of std::sort on the
		// ranges above 16 elements (whole warp, one range after the other), then ONE pass in which every element ranks itself
		// inside its leaf -- the stable order that the insertion sorts of std::sort leave (ncu: the per-lane insertion sorts were
		// 40 % of this kernel's stall samples) -- then the gap flags.
		const int wq = (threadIdx.x >> 5) & 3;
		int *srl = s_tmp[wq], *sscr = srl + WARP_EL_CAP, *sseg = srl + 3 * WARP_EL_CAP;
		unsigned char *sf = s_flag[wq];
		for(int i = lane; i < n; i += 32) sf[i] = (i == 0) ? 1 : 0;
		__syncwarp();
		for(int r = 0; r < 4; r++)
		{
			for(int i = lane; i < n; i += 32) { int32_t fr = (int32_t)(u32)(el[i] & 0xffffffffULL); el[i] = pack_key(pc.key(r, fr), fr); }
			warp_sort_level128(el, n, sf, srl, sscr, sseg, lane);
			for(int i = lane; i < n; i += 32)
				if(i > 0 && !sf[i] && unpack_key(el[i]) - unpack_key(el[i - 1]) > gap) sf[i] = 1;
			__syncwarp();
		}
		for(int i = lane; i < n; i += 32) { members[mo + i] = (int32_t)(u32)(el[i] & 0xffffffffULL); flag[i] = sf[i]; }
		__syncwarp();
		continue;
	}
	for(int i = lane; i < n; i += 32) flag[i] = (i == 0) ? 1 : 0;
	__syncwarp();
	for(int r = 0; r < 4; r++)
	{
		for(int i = lane; i < n; i += 32) { int32_t fr = (int32_t)(u32)(el[i] & 0xffffffffULL); el[i] = pack_key(pc.key(r, fr), fr); }
		// current ranges
		int nr = 0;
		for(int base = 0; base < n; base += 32)
		{
			int i = base + lane;
			bool st = i < n && flag[i];
			unsigned m = __ballot_sync(FULL, st);
			if(st) rl[nr + __popc(m & ((1u << lane) - 1u))] = i;
			nr += __popc(m);
		}
		__syncwarp();
		// big ranges: the whole warp, one after the other
		for(int k = 0; k < nr; k++)
		{
			int lo = rl[k], hi = (k + 1 < nr) ? rl[k + 1] : n;
			if(hi - lo > LANE_RANGE) warp_std_sort(el + lo, hi - lo, less, ss + 3 * lo);
		}
		// small ranges: one lane each
		for(int k = lane; k < nr; k += 32)
		{
			int lo = rl[k], hi = (k + 1 < nr) ? rl[k + 1] : n;
			if(hi - lo <= LANE_RANGE) std_sort_handles(el + lo, hi - lo, less);
		}
		__syncwarp();
		for(int i = lane; i < n; i += 32)
			if(i > 0 && !flag[i] && unpack_key(el[i]) - unpack_key(el[i - 1]) > gap) flag[i] = 1;
		__syncwarp();
	}
	for(int i = lane; i < n; i += 32) members[mo + i] = (int32_t)(u32)(el[i] & 0xffffffffULL);
	__syncwarp();
	}
}
#endif

// diagnostic kernel behind agpu_debug_sort_perm: elements carry (key, original index)
KERNEL k_debug_sort(const int32_t *keys, int n, u64 *el, int32_t *scratch, int32_t *perm)
{
	key_less less;
#ifndef AGPU_EMU
	const int lane = threadIdx.x & 31;
	// the same dispatch as k_group_partition_warp: <= 16 one lane, <= 32 in registers, <= WARP_EL_CAP in shared memory
	__shared__ u64 d_el[WARP_EL_CAP];
	__shared__ int d_tmp[4 * WARP_EL_CAP];
	__shared__ unsigned char d_flag[WARP_EL_CAP];
	for(int i = lane; i < n; i += 32) el[i] = pack_key(keys[i], i);
	__syncwarp();
	if(n <= LANE_RANGE) { if(lane == 0) std_sort_handles(el, n, less); __syncwarp(); }
	else if(n <= 32)
	{
		const bool have = lane < n;
		u64 x = have ? el[lane] : ~0ULL;
		warp_sort_level32(x, have, lane == 0, n, lane, d_el);
		if(have) el[lane] = x;
		__syncwarp();
	}
	else if(n <= WARP_EL_CAP)
	{
		for(int i = lane; i < n; i += 32) { d_el[i] = el[i]; d_flag[i] = i == 0; }
		__syncwarp();
		warp_sort_level128(d_el, n, d_flag, d_tmp, d_tmp + WARP_EL_CAP, d_tmp + 3 * WARP_EL_CAP, lane);
		for(int i = lane; i < n; i += 32) el[i] = d_el[i];
		__syncwarp();
	}
	else warp_std_sort(el, n, less, scratch);
	for(int i = lane; i < n; i += 32) perm[i] = (int32_t)(u32)(el[i] & 0xffffffffULL);
#else
	for(int i = 0; i < n; i++) el[i] = pack_key(keys[i], i);
	std_sort_handles(el, n, less);
	for(int i = 0; i < n; i++) perm[i] = (int32_t)(u32)(el[i] & 0xffffffffULL);
	(void)scratch;
#endif
}

struct clusters_out
{
	int32_t *bounds, *extend, *count, *chain1, *chain2, *bundle;
	int64_t *fr_begin;           // [C+1] member range of the cluster
};

// ---- C4: one thread per member position that starts a cluster (rnacore/graph_cluster.cc:106-165)
KERNEL_OCC(8) k_cluster_emit(int64_t n_mem, const int32_t *cflag_i /* >= 0 at cluster starts, -1 elsewhere */, const int64_t *crank,
		const int32_t *members, const int32_t *mem_bundle_hint, int32_t n_bundles, const int64_t *frg_off, const int64_t *member_boff,
		hits_dev h, const int32_t *f_h1, const int32_t *f_h2, const int32_t *handle_chain, graph_dev g, cluster_dev c, clusters_out o)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_mem) return;
	if(cflag_i[i] < 0) return;
	int64_t cid = crank[i];
	o.fr_begin[cid] = i;
	int b = find_segment(member_boff, n_bundles, i);
	int64_t f0 = frg_off[b], h0 = h.bundle_hit_off[b];
	// extent: up to the next cluster start (every group start is one) or the end of the members
	int64_t j = i + 1;
	while(j < n_mem && cflag_i[j] < 0) j++;
	int cnt = (int)(j - i);
	int32_t fr0 = members[i];
	int64_t a1 = h0 + f_h1[f0 + fr0], a2 = h0 + f_h2[f0 + fr0];
	int32_t b0 = h.pos[a1], b1 = h.rpos[a1], b2 = h.pos[a2], b3 = h.rpos[a2];
	int32_t s0 = 0, s1 = 0, s2 = 0, s3 = 0;
	for(int64_t x = i; x < j; x++)
	{
		int32_t fr = members[x];
		int64_t x1 = h0 + f_h1[f0 + fr], x2 = h0 + f_h2[f0 + fr];
		s0 += h.pos[x1] - b0; s1 += h.rpos[x1] - b1; s2 += h.pos[x2] - b2; s3 += h.rpos[x2] - b3;
	}
	o.bounds[4 * cid] = s0 / cnt + b0; o.bounds[4 * cid + 1] = s1 / cnt + b1;
	o.bounds[4 * cid + 2] = s2 / cnt + b2; o.bounds[4 * cid + 3] = s3 / cnt + b3;
	o.count[cid] = cnt;
	o.chain1[cid] = handle_chain[a1];
	o.chain2[cid] = handle_chain[a2];
	o.bundle[cid] = b;
	gview gv = graph_of(g, b);
	int64_t gf = f0 + fr0;
	o.extend[4 * cid] = gv.v_l[c.m_a1[2 * gf]]; o.extend[4 * cid + 1] = gv.v_r[c.m_a2[2 * gf]];
	o.extend[4 * cid + 2] = gv.v_l[c.m_a1[2 * gf + 1]]; o.extend[4 * cid + 3] = gv.v_r[c.m_a2[2 * gf + 1]];
}

// cflag (0/1) -> -1 / 1 so that the flag-rank scan can be reused
KERNEL k_flag_to_sign(int64_t n, int32_t *v)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	v[i] = v[i] > 0 ? 1 : -1;
}

} // namespace agpu

struct cluster_state
{
	bool built = false;
	// chain paths
	agpu::dbuf<int32_t> cp_valid, cp_mono, cp_first, cp_last, cp_nruns, cp_runs;
	// per fragment
	agpu::dbuf<int32_t> f_ok, m_a1, m_a2, f_next, leader, leader_size;
	agpu::dbuf<agpu::u64> f_hash, slot_word, elems;
	agpu::dbuf<int64_t> f_slot, reg_off, member_off, member_boff, crank, clu_off;
	agpu::dbuf<int32_t> slot_min, slot_n, slot_head, members, cflag, n_big, big_list, part_scratch;
	// clusters
	int64_t n_mem = 0, n_clu = 0;
	agpu::dbuf<int32_t> c_bounds, c_extend, c_count, c_chain1, c_chain2, c_bundle;
	agpu::dbuf<int64_t> c_fr_begin;
	std::vector<int64_t> clu_off_host;

	agpu::chain_paths paths()
	{
		agpu::chain_paths cp;
		cp.valid = cp_valid.p; cp.mono = cp_mono.p; cp.first = cp_first.p; cp.last = cp_last.p; cp.nruns = cp_nruns.p; cp.runs = cp_runs.p;
		return cp;
	}

	agpu::cluster_dev dev()
	{
		agpu::cluster_dev c;
		c.f_ok = f_ok.p; c.m_a1 = m_a1.p; c.m_a2 = m_a2.p; c.f_hash = f_hash.p; c.f_slot = f_slot.p; c.f_next = f_next.p;
		c.reg_off = reg_off.p; c.slot_word = slot_word.p; c.slot_min = slot_min.p; c.slot_n = slot_n.p; c.slot_head = slot_head.p;
		return c;
	}
};

#endif
