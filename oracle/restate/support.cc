// TEST INFRASTRUCTURE ONLY (oracle/).  Restatement of the cross-sample support features of assembler::assemble(vector<bundle*>)
// (meta/assembler.cc:177-373): junction_support (:375-417), non_splicing_support (:419-462), start_end_support (:678-779),
// boundary_extend (:781-880); fix_missing_edges (:946-975) changes nothing and is left out.  Member k is assembled right after its
// own round, and assemble(gr, ps, sid) (:1075-1134) regroups the boundaries of its graph (group_start_boundaries /
// group_end_boundaries, rnacore/graph_reviser.cc:916-1066) before the later members look at it: that is restated too.
// Written over the flat containers of restate.h; the order of the loops is the reference's.
#include "restate.h"

#include <algorithm>
#include <functional>

namespace orc {

// combine_bundles (meta/assembler.cc:152-175) + bundle::combine (meta/bundle.cc:90-107)
void combine_bundles(bundle **bs, int n, bundle &cb, std::vector<int> *order)
{
	const bundle &b0 = *bs[0];
	cb.prm = b0.prm;
	cb.tid = b0.tid; cb.lpos = b0.lpos; cb.rpos = b0.rpos; cb.strand = b0.strand;
	std::vector<std::pair<int, int> > v;
	for(int k = 0; k < n; k++) v.push_back(std::make_pair(k, (int)bs[k]->mmap.segments().size()));
	std::sort(v.begin(), v.end(), [](const std::pair<int, int> &x, const std::pair<int, int> &y) { return x.second > y.second; });
	for(size_t i = 0; i < v.size(); i++)
	{
		const bundle &bb = *bs[v[i].first];
		if(cb.lpos > bb.lpos) cb.lpos = bb.lpos;
		if(cb.rpos < bb.rpos) cb.rpos = bb.rpos;
		cb.hcst.add(bb.hcst);
		cb.fcst.add(bb.fcst);
		cb.mmap.add(bb.mmap);
		if(order) order->push_back(v[i].first);
	}
}

typedef std::pair<int32_t, int32_t> junc_key;
struct junc_val { std::set<int> samples; std::map<int, double> abd; };

static void init_support(const graph &gr, support &s, int sample, std::map<junc_key, junc_val> &jm)
{
	const int ne = (int)gr.edges.size(), n = gr.nv() - 1;
	s.samples.assign(ne, std::set<int>()); s.spabd.assign(ne, std::map<int, double>()); s.abd.assign(ne, 0.0); s.count.assign(ne, 0);
	s.loss.assign(gr.nv(), std::array<double, 4>{{0, 0, 0, 0}});
	for(int e = 0; e < ne; e++)
	{
		if(!gr.edges[e].alive) continue;
		s.samples[e].insert(sample);
		s.spabd[e][sample] = gr.edges[e].w;
		s.abd[e] = gr.edges[e].w;
		s.count[e] = 1;
		const int a = gr.edges[e].s, b = gr.edges[e].t;
		if(a == 0 || b == n) continue;
		if(gr.vr[a] == gr.vl[b]) continue;
		junc_val &jv = jm[junc_key(gr.vr[a], gr.vl[b])];
		jv.samples.insert(sample);
		jv.abd.insert(std::make_pair(sample, gr.edges[e].w));            // the first entry of a sample stays
	}
}

// assembler::junction_support
static void junction_support(const graph &gr, support &s, const std::map<junc_key, junc_val> &jm)
{
	const int n = gr.nv() - 1;
	for(size_t e = 0; e < gr.edges.size(); e++)
	{
		if(!gr.edges[e].alive) continue;
		const int a = gr.edges[e].s, b = gr.edges[e].t;
		if(a == 0 || b == n) continue;
		if(gr.vr[a] == gr.vl[b]) continue;
		std::map<junc_key, junc_val>::const_iterator it = jm.find(junc_key(gr.vr[a], gr.vl[b]));
		if(it == jm.end()) continue;
		s.samples[e] = it->second.samples;
		s.spabd[e] = it->second.abd;
		s.count[e] = (int)s.samples[e].size();
		for(auto &z : it->second.abd) s.abd[e] += z.second;
	}
}

static void credit(support &s, int e, int sample, double w)
{
	s.samples[e].insert(sample);
	s.count[e] = (int)s.samples[e].size();
	s.spabd[e][sample] += w;
	s.abd[e] += w;
}

// assembler::non_splicing_support(sample_id, gr, gx): vertices / edges of gr supporting the adjacent edges of gx
static void non_splicing_support(int sample, const graph &gr, const graph &gx, support &sx)
{
	const int n = gx.nv() - 1;
	for(size_t e = 0; e < gx.edges.size(); e++)
	{
		if(!gx.edges[e].alive) continue;
		const int a = gx.edges[e].s, b = gx.edges[e].t;
		if(a == 0 || b == n) continue;
		if(gx.vr[a] != gx.vl[b]) continue;
		const int32_t p = gx.vl[b];
		const int k1 = gr.locate_vertex(p - 1), k2 = gr.locate_vertex(p);
		if(k1 < 0 || k2 < 0) continue;
		if(k1 == k2) credit(sx, (int)e, sample, gr.vw[k1]);
		else if(gr.vr[k1] == gr.vl[k2] && gr.find_edge(k1, k2) >= 0) credit(sx, (int)e, sample, gr.edges[gr.find_edge(k1, k2)].w);
	}
}

// assembler::start_end_support(sample_id, gr, gx): boundary edges of gr supporting boundary edges of gx
static void start_end_support(int sample, const graph &gr, const graph &gx, support &sx)
{
	const int nr = gr.nv() - 1, nx = gx.nv() - 1;
	for(auto &pr : gr.out[0])
	{
		const int t = pr.first;
		const int32_t p = gr.vr[t];
		int k = gx.locate_vertex(p - 1);
		if(k < 0) continue;
		int eb = gx.find_edge(0, k);
		bool cont = true;
		while(eb < 0)
		{
			k--;
			if(k == 0) { cont = false; break; }
			if(p - gx.vr[k] > 200) cont = false;
			if(gx.vl[k + 1] != gx.vr[k]) cont = false;
			if(gx.find_edge(k, k + 1) < 0) cont = false;
			if(!cont) break;
			eb = gx.find_edge(0, k);
		}
		if(!cont) continue;
		credit(sx, eb, sample, gr.edges[pr.second].w);
	}
	for(auto &pr : gr.in[nr])
	{
		const int s = pr.first;
		const int32_t p = gr.vl[s];
		int k = gx.locate_vertex(p);
		if(k < 0) continue;
		int eb = gx.find_edge(k, nx);
		bool cont = true;
		while(eb < 0)
		{
			k++;
			if(k == nx) { cont = false; break; }
			if(gx.vl[k] - p > 200) cont = false;
			if(gx.vr[k - 1] != gx.vl[k]) cont = false;
			if(gx.find_edge(k - 1, k) < 0) cont = false;
			if(!cont) break;
			eb = gx.find_edge(k, nx);
		}
		if(!cont) continue;
		credit(sx, eb, sample, gr.edges[pr.second].w);
	}
}

static double in_weights(const graph &g, int k) { double w = 0; for(auto &pr : g.in[k]) w += g.edges[pr.second].w; return w; }
static double out_weights(const graph &g, int k) { double w = 0; for(auto &pr : g.out[k]) w += g.edges[pr.second].w; return w; }

// assembler::boundary_extend(sample_id, gr, gx, pos_type): what a boundary of gr would lose inside gx
static void boundary_extend(int sample, const graph &gr, support &sr, const graph &gx, int pos_type)
{
	const int nr = gr.nv() - 1, nx = gx.nv() - 1;
	const int slot = (sample == -1 && pos_type == 1) ? 3 : pos_type - 1;
	for(auto &pr : gr.out[0])
	{
		const int t = pr.first;
		int k = -1;
		if(pos_type == 1) k = gx.locate_vertex(gr.vl[t]);
		else if(pos_type == 2) k = gx.locate_vertex(gr.vr[t] - 1);
		else if(pos_type == 3 && gr.find_edge(t, t + 1) >= 0 && gr.vr[t] == gr.vl[t + 1] && t + 1 < nr) k = gx.locate_vertex(gr.vr[t]);
		if(k <= 0 || gx.find_edge(0, k) >= 0) continue;
		double loss;
		if(gx.find_edge(k - 1, k) >= 0 && gx.vr[k - 1] == gx.vl[k]) loss = in_weights(gx, k) - gx.edges[gx.find_edge(k - 1, k)].w;
		else loss = in_weights(gx, k);
		sr.loss[t][slot] += loss;
	}
	for(auto &pr : gr.in[nr])
	{
		const int s = pr.first;
		int k = -1;
		if(pos_type == 1) k = gx.locate_vertex(gr.vr[s] - 1);
		else if(pos_type == 2) k = gx.locate_vertex(gr.vl[s]);
		else if(pos_type == 3 && s > 1 && gr.find_edge(s - 1, s) >= 0 && gr.vr[s - 1] == gr.vl[s]) k = gx.locate_vertex(gr.vl[s] - 1);
		if(k < 0 || k == nx || gx.find_edge(k, nx) >= 0) continue;
		double loss;
		if(gx.find_edge(k, k + 1) >= 0 && gx.vr[k] == gx.vl[k + 1]) loss = out_weights(gx, k) - gx.edges[gx.find_edge(k, k + 1)].w;
		else loss = out_weights(gx, k);
		sr.loss[s][slot] += loss;
	}
}

// check_continuous_vertices (rnacore/essential.cc:436-446)
static bool continuous(const graph &gr, int x, int y)
{
	for(int i = x; i < y; i++)
	{
		if(gr.find_edge(i, i + 1) < 0) return false;
		if(gr.vr[i] != gr.vl[i + 1]) return false;
	}
	return true;
}

// group_start_boundaries / group_end_boundaries (rnacore/graph_reviser.cc:916-1066) as far as they change the graph: start (end)
// boundaries of one continuous stretch within max_group_boundary_distance collapse onto the first (last) one
static void group_boundaries(graph &gr, int32_t max_dist)
{
	const int n = gr.nv() - 1;
	std::vector<int> v;
	for(auto &pr : gr.out[0]) v.push_back(pr.first);
	if(v.size() > 1)
	{
		std::sort(v.begin(), v.end());
		int32_t p2 = gr.vl[v[0]];
		int k1 = v[0], k2 = v[0];
		int ea = gr.find_edge(0, v[0]);
		double wa = gr.edges[ea].w;
		for(size_t i = 1; i < v.size(); i++)
		{
			const int32_t p = gr.vl[v[i]];
			const int eb = gr.find_edge(0, v[i]);
			const double wb = gr.edges[eb].w;
			bool b = continuous(gr, k2, v[i]);
			if(p - p2 > max_dist) b = false;
			if(!b) { p2 = p; k1 = v[i]; k2 = v[i]; ea = eb; wa = wb; continue; }
			for(int j = k1; j < v[i]; j++)
			{
				const int ec = gr.find_edge(j, j + 1);
				const double vc = gr.vw[j], wc = gr.edges[ec].w;
				gr.vw[j] = vc + wb;
				gr.edges[ec].w = wc + wb;
			}
			wa += wb;
			gr.edges[ea].w = wa;
			gr.remove_edge(eb);
			k2 = v[i];
			p2 = p;
		}
	}
	v.clear();
	for(auto &pr : gr.in[n]) v.push_back(pr.first);
	if(v.size() > 1)
	{
		std::sort(v.begin(), v.end(), std::greater<int>());
		int32_t p2 = gr.vr[v[0]];
		int k1 = v[0], k2 = v[0];
		int ea = gr.find_edge(v[0], n);
		double wa = gr.edges[ea].w;
		for(size_t i = 1; i < v.size(); i++)
		{
			const int32_t p = gr.vr[v[i]];
			const int eb = gr.find_edge(v[i], n);
			const double wb = gr.edges[eb].w;
			bool b = continuous(gr, v[i], k2);
			if(p2 - p > max_dist) b = false;
			if(!b) { p2 = p; k1 = v[i]; k2 = v[i]; ea = eb; wa = wb; continue; }
			for(int j = v[i]; j < k1; j++)
			{
				const int ec = gr.find_edge(j, j + 1);
				const double wc = gr.edges[ec].w;
				gr.edges[ec].w = wc + wb;
				gr.vw[j + 1] = wc + wb;          // as the reference writes it: the edge's new weight, not the vertex's own plus wb
			}
			wa += wb;
			gr.edges[ea].w = wa;
			gr.remove_edge(eb);
			k2 = v[i];
			p2 = p;
		}
	}
}

int group_support(bundle **bs, int n, std::vector<graph> &grs, std::vector<support> &sups, graph &gx, support &sx)
{
	bundle cb;
	combine_bundles(bs, n, cb, NULL);
	builder_out bo;
	build_graph(cb, gx, bo);
	if(bo.repeated_bounds) return -1;
	std::map<junc_key, junc_val> jm;
	init_support(gx, sx, -1, jm);
	std::vector<graph> live(n);                           // the graphs as the rounds see them (regrouped once assembled)
	grs.assign(n, graph()); sups.assign(n, support());
	for(int k = 0; k < n; k++)
	{
		builder_out bk;
		build_graph(*bs[k], live[k], bk);
		if(bk.repeated_bounds) return -1;
		revision rv;
		revise_graph(*bs[k], live[k], rv);
		init_support(live[k], sups[k], bs[k]->sample, jm);
	}
	for(int k = 0; k < n; k++)
	{
		junction_support(live[k], sups[k], jm);
		for(int j = 0; j < n; j++)
		{
			start_end_support(bs[j]->sample, live[j], live[k], sups[k]);
			non_splicing_support(bs[j]->sample, live[j], live[k], sups[k]);
			for(int t = 1; t <= 3; t++) boundary_extend(bs[j]->sample, live[k], sups[k], live[j], t);
		}
		start_end_support(bs[k]->sample, live[k], gx, sx);
		non_splicing_support(bs[k]->sample, live[k], gx, sx);
		boundary_extend(-1, live[k], sups[k], gx, 1);
		grs[k] = live[k];                                 // what the reference hands to assemble(gr, ps, sid) ...
		group_boundaries(live[k], bs[0]->prm.max_group_boundary_distance);   // ... which regroups its boundaries (util/parameters.cc:77)
	}
	junction_support(gx, sx, jm);
	return 0;
}

} // namespace orc
