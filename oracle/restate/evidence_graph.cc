// TEST INFRASTRUCTURE ONLY (oracle/): restatement of the evidence store and the splice-graph builder.
#include "restate.h"

#include <algorithm>
#include <cmath>
#include <cstdio>

namespace orc {

// ---- chain_set (rnacore/chain_set.cc:24-123, :187-210) -----------------------------------------------
void chain_set::add(const chain_t &v, const AI3 &a)
{
	if(v.empty()) return;
	std::map<int32_t, int>::iterator it = pmap.find(v[0]);
	if(it == pmap.end())
	{
		chains.push_back(std::vector<std::pair<chain_t, AI3> >(1, std::make_pair(v, a)));
		pmap[v[0]] = (int)chains.size() - 1;
		return;
	}
	std::vector<std::pair<chain_t, AI3> > &vv = chains[it->second];
	for(size_t i = 0; i < vv.size(); i++)
	{
		if(vv[i].first != v) continue;
		for(int k = 0; k < 3; k++) vv[i].second[k] += a[k];
		return;
	}
	vv.push_back(std::make_pair(v, a));
}

void chain_set::add(const chain_t &v, int h, char c)
{
	if(v.empty()) return;
	if(h >= 0 && hmap.count(h)) return;
	int xs = (c == '+') ? 1 : ((c == '-') ? 2 : 0);
	AI3 one = {0, 0, 0};
	one[xs] = 1;
	std::map<int32_t, int>::iterator it = pmap.find(v[0]);
	if(it == pmap.end())
	{
		chains.push_back(std::vector<std::pair<chain_t, AI3> >(1, std::make_pair(v, one)));
		int n = (int)chains.size() - 1;
		pmap[v[0]] = n;
		if(h >= 0) hmap[h] = AI3({n, 0, xs});
		return;
	}
	int k = it->second;
	std::vector<std::pair<chain_t, AI3> > &vv = chains[k];
	for(size_t i = 0; i < vv.size(); i++)
	{
		if(vv[i].first != v) continue;
		if(h >= 0) hmap[h] = AI3({k, (int)i, xs});
		vv[i].second[xs]++;
		return;
	}
	vv.push_back(std::make_pair(v, one));
	if(h >= 0) hmap[h] = AI3({k, (int)vv.size() - 1, xs});
}

void chain_set::add(const chain_set &cs)
{
	for(size_t i = 0; i < cs.chains.size(); i++)
		for(size_t j = 0; j < cs.chains[i].size(); j++) add(cs.chains[i][j].first, cs.chains[i][j].second);
}

const chain_t *chain_set::get(int h) const
{
	std::map<int, AI3>::const_iterator it = hmap.find(h);
	if(h < 0 || it == hmap.end()) return NULL;
	return &chains[it->second[0]][it->second[1]].first;
}

std::vector<int32_t> chain_set::get_splices() const
{
	std::set<int32_t> s;
	for(size_t i = 0; i < chains.size(); i++)
		for(size_t j = 0; j < chains[i].size(); j++)
		{
			const AI3 &a = chains[i][j].second;
			if(a[0] + a[1] + a[2] <= 0) continue;
			s.insert(chains[i][j].first.begin(), chains[i][j].first.end());
		}
	return std::vector<int32_t>(s.begin(), s.end());
}

// ---- coverage map ---------------------------------------------------------------------------------------
void coverage_map::add(int32_t l, int32_t r, int32_t v)
{
	if(l >= r || v == 0) return;       // empty interval / identity value: no-op under partial_absorber
	delta[l] += v;                     // operator[] creates the border even when the deltas cancel
	delta[r] -= v;
}

void coverage_map::add(const coverage_map &m)
{
	std::vector<seg> s = m.segments();
	for(size_t i = 0; i < s.size(); i++) add(s[i].l, s[i].r, s[i].c);
}

std::vector<coverage_map::seg> coverage_map::segments() const
{
	std::vector<seg> out;
	int32_t cov = 0;
	for(std::map<int32_t, int32_t>::const_iterator it = delta.begin(); it != delta.end(); ++it)
	{
		cov += it->second;
		std::map<int32_t, int32_t>::const_iterator nx = it;
		++nx;
		if(nx == delta.end()) break;
		if(cov > 0) { seg s = {it->first, nx->first, cov}; out.push_back(s); }
	}
	return out;
}

// ---- graph container ------------------------------------------------------------------------------------
int graph::add_edge(int s, int t, double w, int st)
{
	edge e = {s, t, w, st, true};
	edges.push_back(e);
	int k = (int)edges.size() - 1;
	out[s].insert(std::make_pair(t, k));
	in[t].insert(std::make_pair(s, k));
	return k;
}

void graph::remove_edge(int e)
{
	if(!edges[e].alive) return;
	edges[e].alive = false;
	out[edges[e].s].erase(std::make_pair(edges[e].t, e));
	in[edges[e].t].erase(std::make_pair(edges[e].s, e));
}

int graph::find_edge(int s, int t) const
{
	std::set<std::pair<int, int> >::const_iterator it = out[s].lower_bound(std::make_pair(t, -1));
	if(it == out[s].end() || it->first != t) return -1;
	return it->second;
}

// splice_graph::build_vertex_index (rnacore/splice_graph.cc:1087-1099)
void graph::build_vertex_index()
{
	lindex.clear(); rindex.clear();
	int n = nv() - 1;
	for(int i = 0; i <= n; i++)
	{
		if(i != 0) lindex.insert(std::make_pair(vl[i], i));
		if(i != n) rindex.insert(std::make_pair(vr[i], i));
	}
}

// splice_graph::locate_vertex (rnacore/splice_graph.cc:1166-1215)
int graph::locate_vertex(int32_t p) const
{
	int a = 1, b = nv() - 1;
	int m = -1;
	while(a < b)
	{
		int mid = (a + b) / 2;
		if(p >= vl[mid] && p < vr[mid]) { m = mid; break; }
		if(p < vl[mid]) b = mid;
		else a = mid + 1;
	}
	if(m < 0) m = b;
	if(p >= vl[m] && p < vr[m]) return m;
	return -1;
}

// ---- regions -> partial exons ---------------------------------------------------------------------------
namespace {

enum { START_BOUNDARY = 1, END_BOUNDARY = 2, LEFT_SPLICE = 3, RIGHT_SPLICE = 4, LEFT_RIGHT_SPLICE = 5 };

typedef std::vector<coverage_map::seg> segs_t;

// locate_boundary_iterators (rnacore/interval_map.cc:70-87): segments lying fully inside [x, y)
bool inside(const segs_t &s, int32_t x, int32_t y, int &i0, int &i1)
{
	int n = (int)s.size();
	i0 = 0;
	while(i0 < n && s[i0].l < x) i0++;
	if(i0 >= n || s[i0].r > y) return false;
	i1 = n - 1;
	while(i1 >= 0 && s[i1].r > y) i1--;
	if(i1 < 0 || s[i1].l < x) return false;
	return i0 <= i1;
}

// evaluate_rectangle (rnacore/interval_map.cc:166-195)
void evaluate_rectangle(const segs_t &s, int32_t ll, int32_t rr, double &ave, double &dev, double &mx)
{
	ave = 0; dev = 1; mx = 0;
	int i0, i1;
	if(!inside(s, ll, rr, i0, i1)) return;
	int32_t sum = 0, m = 0;
	for(int i = i0; i <= i1; i++)
	{
		sum = (int32_t)((uint32_t)sum + (uint32_t)((s[i].r - s[i].l) * s[i].c));
		if(s[i].c > m) m = s[i].c;
	}
	mx = 1.0 * m;
	ave = 1.0 * sum / (rr - ll);
	double var = 0;
	for(int i = i0; i <= i1; i++) var += (s[i].c - ave) * (s[i].c - ave) * (s[i].r - s[i].l);
	dev = sqrt(var / (rr - ll));
}

// region::empty_subregion (rnacore/region.cc:88-107)
bool empty_subregion(const segs_t &s, int32_t p1, int32_t p2, const orc_params &prm)
{
	if(p2 - p1 < prm.min_subregion_length) return true;
	int i0, i1;
	if(!inside(s, p1, p2, i0, i1)) return true;
	int32_t sum = 0;
	for(int i = i0; i <= i1; i++) sum = (int32_t)((uint32_t)sum + (uint32_t)((s[i].r - s[i].l) * s[i].c));
	double ratio = sum * 1.0 / (p2 - p1);
	return ratio < prm.min_subregion_overlap;
}

// region::region (rnacore/region.cc:22-169) on the local segment list of the bundle
void region_pexons(const segs_t &s, int32_t lpos, int32_t rpos, int ltype, int rtype, const orc_params &prm, std::vector<pexon> &out)
{
	// build_join_interval_map: maximal runs of touching segments inside the region
	std::vector<std::pair<int32_t, int32_t> > runs;
	int i0, i1;
	if(inside(s, lpos, rpos, i0, i1))
	{
		for(int i = i0; i <= i1; i++)
		{
			if(!runs.empty() && runs.back().second == s[i].l) runs.back().second = s[i].r;
			else runs.push_back(std::make_pair(s[i].l, s[i].r));
		}
	}
	// smooth_join_interval_map (only between two splice ends)
	if(ltype == RIGHT_SPLICE && rtype == LEFT_SPLICE)
	{
		std::vector<std::pair<int32_t, int32_t> > fill;
		int32_t p = lpos;
		for(size_t k = 0; k < runs.size(); k++)
		{
			if(runs[k].first - p <= prm.min_subregion_gap) fill.push_back(std::make_pair(p, runs[k].first));
			p = runs[k].second;
		}
		if(p < rpos && rpos - p <= prm.min_subregion_gap) fill.push_back(std::make_pair(p, rpos));
		for(size_t k = 0; k < fill.size(); k++) if(fill[k].first < fill[k].second) runs.push_back(fill[k]);
		std::sort(runs.begin(), runs.end());
		std::vector<std::pair<int32_t, int32_t> > joined;
		for(size_t k = 0; k < runs.size(); k++)
		{
			if(!joined.empty() && joined.back().second == runs[k].first) joined.back().second = runs[k].second;
			else joined.push_back(runs[k]);
		}
		runs.swap(joined);
	}
	// build_partial_exons
	pexon stub = {0, 0, 0, 0, prm.min_guaranteed_edge_weight, 1.0, -1.0, 0, true, false};
	if(runs.empty() && rpos == lpos + 1 && (ltype == END_BOUNDARY || rtype == START_BOUNDARY))
	{
		stub.lpos = lpos; stub.rpos = rpos; stub.ltype = ltype; stub.rtype = rtype;
		out.push_back(stub);
		return;
	}
	if(!runs.empty() && runs[0].first == lpos && runs[0].second == rpos)
	{
		pexon pe = {lpos, rpos, ltype, rtype, 0, 0, 0, 0, false, false};
		evaluate_rectangle(s, lpos, rpos, pe.ave, pe.dev, pe.max);
		out.push_back(pe);
		return;
	}
	if(ltype == RIGHT_SPLICE && (runs.empty() || runs[0].first != lpos))
	{
		stub.lpos = lpos; stub.rpos = lpos + 1; stub.ltype = ltype; stub.rtype = END_BOUNDARY;
		out.push_back(stub);
	}
	for(size_t k = 0; k < runs.size(); k++)
	{
		int32_t p1 = runs[k].first, p2 = runs[k].second;
		bool b = empty_subregion(s, p1, p2, prm);
		if(p1 == lpos && ltype == RIGHT_SPLICE) b = false;
		if(p2 == rpos && rtype == LEFT_SPLICE) b = false;
		if(b) continue;
		pexon pe = {p1, p2, (p1 == lpos) ? ltype : START_BOUNDARY, (p2 == rpos) ? rtype : END_BOUNDARY, 0, 0, 0, 0, false, false};
		evaluate_rectangle(s, p1, p2, pe.ave, pe.dev, pe.max);
		out.push_back(pe);
	}
	if(rtype == LEFT_SPLICE && (runs.empty() || runs.back().second != rpos))
	{
		stub.lpos = rpos - 1; stub.rpos = rpos; stub.ltype = START_BOUNDARY; stub.rtype = rtype;
		out.push_back(stub);
	}
}

} // namespace

// graph_builder::build (rnacore/graph_builder.cc:24-35)
void build_graph(const bundle &bd, graph &gr, builder_out &bo)
{
	const orc_params &prm = bd.prm;
	std::vector<junction> &junctions = bo.junctions;
	std::vector<pexon> &pexons = bo.pexons;
	junctions.clear(); pexons.clear();

	// build_junctions (:46-125): every chain of hcst, then of fcst, exploded into a temporary chain set
	chain_set jcst;
	const chain_set *src[2] = {&bd.hcst, &bd.fcst};
	for(int w = 0; w < 2; w++)
		for(size_t i = 0; i < src[w]->chains.size(); i++)
			for(size_t j = 0; j < src[w]->chains[i].size(); j++)
			{
				const chain_t &v = src[w]->chains[i][j].first;
				if(v.empty() || v.size() % 2 != 0) continue;
				for(size_t k = 0; k < v.size() / 2; k++)
				{
					chain_t z(2);
					z[0] = v[2 * k]; z[1] = v[2 * k + 1];
					jcst.add(z, src[w]->chains[i][j].second);
				}
			}
	for(size_t i = 0; i < jcst.chains.size(); i++)
		for(size_t j = 0; j < jcst.chains[i].size(); j++)
		{
			const chain_t &v = jcst.chains[i][j].first;
			const AI3 &a = jcst.chains[i][j].second;
			if(v.size() != 2 || v[0] >= v[1]) continue;
			int count = a[0] + a[1] + a[2];
			if(count < prm.min_junction_support) continue;
			junction jc = {v[0], v[1], count, a[0], a[1], a[2], '.', -1, -1};
			if(a[1] > a[2]) jc.strand = '+';
			else if(a[1] < a[2]) jc.strand = '-';
			junctions.push_back(jc);
		}
	// remove_opposite_junctions (:128-175): junction::nm is 0 for every junction (rnacore/junction.cc:26), so both
	// nm / count ratios are 0.0, the strict '<' / '>' tests fail and nothing is ever removed.

	// build_regions (:177-224)
	std::map<int32_t, int> s;
	s.insert(std::make_pair(bd.lpos, (int)START_BOUNDARY));
	s.insert(std::make_pair(bd.rpos, (int)END_BOUNDARY));
	for(size_t i = 0; i < junctions.size(); i++)
	{
		int32_t l = junctions[i].lpos, r = junctions[i].rpos;
		if(s.find(l) == s.end()) s[l] = LEFT_SPLICE;
		else if(s[l] == RIGHT_SPLICE) s[l] = LEFT_RIGHT_SPLICE;
		if(s.find(r) == s.end()) s[r] = RIGHT_SPLICE;
		else if(s[r] == LEFT_SPLICE) s[r] = LEFT_RIGHT_SPLICE;
	}
	std::vector<std::pair<int32_t, int> > v(s.begin(), s.end());
	segs_t segs = bd.mmap.segments();
	for(size_t k = 0; k + 1 < v.size(); k++)
	{
		int lt = v[k].second, rt = v[k + 1].second;
		if(lt == LEFT_RIGHT_SPLICE) lt = RIGHT_SPLICE;
		if(rt == LEFT_RIGHT_SPLICE) rt = LEFT_SPLICE;
		region_pexons(segs, v[k].first, v[k + 1].first, lt, rt, prm, pexons);      // build_partial_exons (:226-242)
	}
	for(size_t i = 0; i < pexons.size(); i++)
	{
		pexon &pe = pexons[i];
		pe.regional = ((pe.lpos != bd.lpos || pe.rpos != bd.rpos) && pe.ltype == START_BOUNDARY && pe.rtype == END_BOUNDARY);
	}

	// classify_partial_exons (:477-514)
	std::map<std::pair<int32_t, int32_t>, int> mj;
	for(size_t i = 0; i < junctions.size(); i++) mj[std::make_pair(junctions[i].lpos, junctions[i].rpos)] = (int)i;
	for(size_t i = 0; i < pexons.size(); i++)
	{
		pexon &pe = pexons[i];
		bool b = false;
		if(pe.lpos == bd.lpos) b = true;
		if(pe.rpos == bd.rpos) b = true;
		if(pe.ltype == RIGHT_SPLICE) b = true;
		if(pe.rtype == LEFT_SPLICE) b = true;
		if(pe.ltype == LEFT_SPLICE && pe.rtype == RIGHT_SPLICE)
		{
			std::map<std::pair<int32_t, int32_t>, int>::iterator it = mj.find(std::make_pair(pe.lpos, pe.rpos));
			if(it == mj.end()) b = true;
			else if(junctions[it->second].count < pe.ave) b = true;
		}
		pe.pvalue = b ? 0 : 1;
	}

	// link_partial_exons (:244-297): the reference asserts that no two partial exons share a bound (:255-258) before it
	// inserts them into its maps; a 1-bp region between a junction end and a junction start with no coverage and
	// min_subregion_gap 0 gets both stubs of build_partial_exons, [p, p + 1) twice
	std::map<int32_t, int> lm, rm;
	bo.repeated_bounds = 0;
	for(size_t i = 0; i < pexons.size(); i++)
	{
		if(!lm.insert(std::make_pair(pexons[i].lpos, (int)i)).second) bo.repeated_bounds++;
		if(!rm.insert(std::make_pair(pexons[i].rpos, (int)i)).second) bo.repeated_bounds++;
	}
	for(size_t i = 0; i < junctions.size(); i++)
	{
		std::map<int32_t, int>::iterator li = rm.find(junctions[i].lpos), ri = lm.find(junctions[i].rpos);
		if(li != rm.end() && ri != lm.end()) { junctions[i].lexon = li->second; junctions[i].rexon = ri->second; }
	}

	// build_splice_graph (:299-426)
	int np = (int)pexons.size(), nv = np + 2;
	gr = graph();
	gr.strand = bd.strand;
	gr.vl.assign(nv, 0); gr.vr.assign(nv, 0); gr.vlen.assign(nv, 0); gr.vtype.assign(nv, 0); gr.vregional.assign(nv, 0);
	gr.vw.assign(nv, 0); gr.vdev.assign(nv, 1.0); gr.vmax.assign(nv, 0);
	gr.out.resize(nv); gr.in.resize(nv);
	gr.vl[0] = gr.vr[0] = bd.lpos;
	gr.vl[nv - 1] = gr.vr[nv - 1] = bd.rpos;
	for(int i = 0; i < np; i++)
	{
		const pexon &r = pexons[i];
		double w = r.ave;
		if(w < prm.min_guaranteed_edge_weight) w = prm.min_guaranteed_edge_weight;
		gr.vl[i + 1] = r.lpos; gr.vr[i + 1] = r.rpos; gr.vlen[i + 1] = r.rpos - r.lpos;
		gr.vtype[i + 1] = (r.pvalue < 0.5) ? 0 : 1;
		gr.vregional[i + 1] = r.regional ? 1 : 0;
		gr.vw[i + 1] = w; gr.vdev[i + 1] = r.dev; gr.vmax[i + 1] = r.max;
	}
	for(size_t i = 0; i < junctions.size(); i++)
	{
		const junction &b = junctions[i];
		if(b.lexon < 0 || b.rexon < 0) continue;
		gr.add_edge(b.lexon + 1, b.rexon + 1, b.count, b.strand == '+' ? 1 : (b.strand == '-' ? 2 : 0));
	}
	for(int i = 0; i < np; i++)
	{
		const pexon &r = pexons[i];
		if(r.ltype == START_BOUNDARY)
		{
			double w = r.ave;
			if(i >= 1 && pexons[i - 1].rpos == r.lpos) w -= pexons[i - 1].ave;
			if(w < prm.min_guaranteed_edge_weight) w = prm.min_guaranteed_edge_weight;
			gr.add_edge(0, i + 1, w, 0);
		}
		if(r.rtype == END_BOUNDARY)
		{
			double w = r.ave;
			if(i < np - 1 && pexons[i + 1].lpos == r.rpos) w -= pexons[i + 1].ave;
			if(w < prm.min_guaranteed_edge_weight) w = prm.min_guaranteed_edge_weight;
			gr.add_edge(i + 1, np + 1, w, 0);
		}
	}
	for(int i = 0; i < np - 1; i++)
	{
		const pexon &x = pexons[i], &y = pexons[i + 1];
		if(x.rpos != y.lpos) continue;
		int xd = (int)gr.out[i + 1].size(), yd = (int)gr.in[i + 2].size();
		double wt = x.ave;
		if(xd < yd) wt = x.ave;
		else if(xd > yd) wt = y.ave;
		else if(x.ave < y.ave) wt = x.ave;
		else if(x.ave > y.ave) wt = y.ave;
		if(wt < prm.min_guaranteed_edge_weight) wt = prm.min_guaranteed_edge_weight;
		gr.add_edge(i + 1, i + 2, wt, 0);
	}

	// refine_splice_graph (rnacore/graph_reviser.cc:899-914)
	while(true)
	{
		bool b = false;
		for(int i = 1; i < nv - 1; i++)
		{
			if(gr.in[i].size() + gr.out[i].size() == 0) continue;
			if(gr.in[i].size() >= 1 && gr.out[i].size() >= 1) continue;
			std::vector<int> kill;
			for(std::set<std::pair<int, int> >::iterator it = gr.in[i].begin(); it != gr.in[i].end(); ++it) kill.push_back(it->second);
			for(std::set<std::pair<int, int> >::iterator it = gr.out[i].begin(); it != gr.out[i].end(); ++it) kill.push_back(it->second);
			for(size_t k = 0; k < kill.size(); k++) gr.remove_edge(kill[k]);
			b = true;
		}
		if(!b) break;
	}
	gr.build_vertex_index();
}

} // namespace orc
