// TEST INFRASTRUCTURE ONLY (oracle/): flat C interface of the restatement (orc_api.h, prefix "orc_") and the
// dumps into named arrays, in the same layout as oracle/ref_driver.cc.
#include "restate.h"
#include "../orc_bag.h"

#include <algorithm>
#include <cstdio>

using namespace orc;

namespace {

void dump_chain_set(const chain_set &cs, orc_bag &bag, const std::string &pre, int nh, const std::string &hname)
{
	std::vector<int32_t> &off = bag.ints(pre + "_off"), &val = bag.ints(pre + "_val"), &cnt = bag.ints(pre + "_cnt"), &grp = bag.ints(pre + "_grp");
	off.clear(); val.clear(); cnt.clear(); grp.clear();
	std::vector<std::vector<int> > flat(cs.chains.size());
	off.push_back(0);
	int c = 0;
	for(size_t i = 0; i < cs.chains.size(); i++)
		for(size_t j = 0; j < cs.chains[i].size(); j++)
		{
			val.insert(val.end(), cs.chains[i][j].first.begin(), cs.chains[i][j].first.end());
			off.push_back((int32_t)val.size());
			for(int k = 0; k < 3; k++) cnt.push_back(cs.chains[i][j].second[k]);
			grp.push_back((int32_t)i);
			flat[i].push_back(c++);
		}
	std::vector<int32_t> &hc = bag.ints(hname), &hx = bag.ints(hname + "_xs");
	hc.assign(nh, -1); hx.assign(nh, -1);
	for(std::map<int, AI3>::const_iterator it = cs.hmap.begin(); it != cs.hmap.end(); ++it)
	{
		if(it->first < 0 || it->first >= nh) continue;
		hc[it->first] = flat[it->second[0]][it->second[1]];
		hx[it->first] = it->second[2];
	}
}

void dump_segments(const coverage_map &m, orc_bag &bag, const std::string &name)
{
	std::vector<int32_t> &seg = bag.ints(name);
	seg.clear();
	std::vector<coverage_map::seg> s = m.segments();
	for(size_t i = 0; i < s.size(); i++) { seg.push_back(s[i].l); seg.push_back(s[i].r); seg.push_back(s[i].c); }
}

void dump_frgs(const bundle &bd, orc_bag &bag, const std::string &name)
{
	std::vector<int32_t> &f = bag.ints(name);
	f.clear();
	for(size_t i = 0; i < bd.frgs.size(); i++) for(int k = 0; k < 3; k++) f.push_back(bd.frgs[i][k]);
}

void dump_builder(const builder_out &bo, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &jc = bag.ints(pre + "junc"), &pe = bag.ints(pre + "pexon");
	std::vector<double> &pd = bag.reals(pre + "pexon_d");
	jc.clear(); pe.clear(); pd.clear();
	for(size_t i = 0; i < bo.junctions.size(); i++)
	{
		const junction &j = bo.junctions[i];
		int32_t row[9] = {j.lpos, j.rpos, j.count, j.xs0, j.xs1, j.xs2, (int32_t)j.strand, j.lexon, j.rexon};
		jc.insert(jc.end(), row, row + 9);
	}
	for(size_t i = 0; i < bo.pexons.size(); i++)
	{
		const pexon &p = bo.pexons[i];
		int32_t row[5] = {p.lpos, p.rpos, p.ltype, p.rtype, p.regional ? 1 : 0};
		pe.insert(pe.end(), row, row + 5);
		pd.push_back(p.ave); pd.push_back(p.dev); pd.push_back(p.stub ? -1.0 : p.max); pd.push_back(p.pvalue);
	}
}

void dump_graph(const graph &gr, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &vi = bag.ints(pre + "vert"), &ei = bag.ints(pre + "edge"), &gs = bag.ints(pre + "graph");
	std::vector<double> &vd = bag.reals(pre + "vert_d"), &ed = bag.reals(pre + "edge_d");
	vi.clear(); vd.clear(); ei.clear(); ed.clear(); gs.clear();
	for(int i = 0; i < gr.nv(); i++)
	{
		int32_t row[5] = {gr.vl[i], gr.vr[i], gr.vlen[i], gr.vtype[i], gr.vregional[i]};
		vi.insert(vi.end(), row, row + 5);
		vd.push_back(gr.vw[i]); vd.push_back(gr.vdev[i]); vd.push_back(gr.vmax[i]);
	}
	for(int i = 0; i < gr.nv(); i++)
		for(std::set<std::pair<int, int> >::const_iterator it = gr.out[i].begin(); it != gr.out[i].end(); ++it)
		{
			const edge &e = gr.edges[it->second];
			ei.push_back(e.s); ei.push_back(e.t); ei.push_back(e.strand);
			ed.push_back(e.w);
		}
	gs.push_back((int32_t)gr.strand);
}

void dump_clusters(const std::vector<cluster> &vc, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &bo = bag.ints(pre + "clu_bounds"), &ex = bag.ints(pre + "clu_extend"), &ct = bag.ints(pre + "clu_count");
	std::vector<int32_t> &o1 = bag.ints(pre + "clu_c1_off"), &v1 = bag.ints(pre + "clu_c1_val"), &o2 = bag.ints(pre + "clu_c2_off"), &v2 = bag.ints(pre + "clu_c2_val");
	std::vector<int32_t> &of = bag.ints(pre + "clu_fr_off"), &vf = bag.ints(pre + "clu_fr_val");
	bo.clear(); ex.clear(); ct.clear(); o1.clear(); v1.clear(); o2.clear(); v2.clear(); of.clear(); vf.clear();
	o1.push_back(0); o2.push_back(0); of.push_back(0);
	for(size_t i = 0; i < vc.size(); i++)
	{
		const cluster &pc = vc[i];
		bo.insert(bo.end(), pc.bounds.begin(), pc.bounds.end());
		ex.insert(ex.end(), pc.extend.begin(), pc.extend.end());
		ct.push_back(pc.count);
		v1.insert(v1.end(), pc.chain1.begin(), pc.chain1.end()); o1.push_back((int32_t)v1.size());
		v2.insert(v2.end(), pc.chain2.begin(), pc.chain2.end()); o2.push_back((int32_t)v2.size());
		vf.insert(vf.end(), pc.frlist.begin(), pc.frlist.end()); of.push_back((int32_t)vf.size());
	}
}

void dump_opt(const std::vector<bridge_path> &opt, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &o = bag.ints(pre + "opt"), &co = bag.ints(pre + "opt_chain_off"), &cv = bag.ints(pre + "opt_chain_val");
	std::vector<int32_t> &wo = bag.ints(pre + "opt_whole_off"), &wv = bag.ints(pre + "opt_whole_val");
	std::vector<double> &os = bag.reals(pre + "opt_score");
	o.clear(); os.clear(); co.clear(); cv.clear(); wo.clear(); wv.clear();
	co.push_back(0); wo.push_back(0);
	for(size_t i = 0; i < opt.size(); i++)
	{
		const bridge_path &p = opt[i];
		o.push_back(p.type); o.push_back(p.strand); o.push_back(p.choices);
		os.push_back(p.score);
		cv.insert(cv.end(), p.chain.begin(), p.chain.end()); co.push_back((int32_t)cv.size());
		wv.insert(wv.end(), p.whole.begin(), p.whole.end()); wo.push_back((int32_t)wv.size());
	}
}

// meta/bundle.cc:66-79 / meta/assembler.cc:989-1012
int cluster_solve_update(graph &gr, bundle &bd, const orc_params &prm, orc_bag &bag, const std::string &pre, bool skip_if_empty)
{
	std::vector<cluster> vc;
	cluster_fragments(gr, bd, vc);
	dump_frgs(bd, bag, pre + "frgs_clustered");
	dump_clusters(vc, bag, pre);
	int cnt = 0;
	if(skip_if_empty && vc.empty()) dump_opt(std::vector<bridge_path>(), bag, pre);
	else
	{
		std::vector<bridge_path> opt;
		bridge_clusters(gr, vc, prm, opt);
		dump_opt(opt, bag, pre);
		for(size_t k = 0; k < vc.size(); k++)
		{
			if(opt[k].type <= 0) continue;
			cnt += update_bridges(bd, vc[k].frlist, opt[k].chain, opt[k].strand);
		}
	}
	dump_frgs(bd, bag, pre + "frgs");
	dump_chain_set(bd.fcst, bag, pre + "fcst", (int)bd.frgs.size(), pre + "frg_chain");
	dump_segments(bd.mmap, bag, pre + "seg");
	std::vector<int32_t> &bc = bag.ints(pre + "bridged");
	bc.assign(1, cnt);
	return cnt;
}

} // namespace

extern "C" {

// bundle_base::add_hit_intervals per hit (rnacore/bundle_base.cc:33-47) + generator::generate (meta/generator.cc:203-227)
void *orc_bundle_new(const orc_bundle_in *in, const orc_params *prm)
{
	bundle *bd = new bundle;
	bd->prm = *prm;
	bd->tid = -1; bd->lpos = 1 << 30; bd->rpos = 0; bd->strand = '.';
	for(int i = 0; i < in->n_hits; i++)
	{
		hit h;
		h.pos = in->pos[i]; h.mpos = in->mpos[i]; h.isize = in->isize[i]; h.flag = in->flag[i];
		h.strand = (char)in->strand[i]; h.xs = (char)in->xs[i]; h.qid = in->qid[i];
		const uint32_t *cig = in->cigar + in->cigar_off[i];
		int nc = (int)(in->cigar_off[i + 1] - in->cigar_off[i]);
		// hit::hit (rnacore/hit.cc:52-65): rpos = pos + bam_cigar2rlen
		int32_t p = h.pos;
		for(int k = 0; k < nc; k++) if((0x3C1A7 >> ((cig[k] & 0xf) << 1)) & 2) p += (int32_t)(cig[k] >> 4);
		h.rpos = p;
		// add_hit (:73-104)
		if(!bd->hits.empty() && bd->hits.back().pos == h.pos && bd->hits.back().rpos == h.rpos) continue;
		bd->hits.push_back(h);
		bd->input_index.push_back(i);
		if(h.pos < bd->lpos) bd->lpos = h.pos;
		int32_t q = h.rpos;
		if(h.mpos > h.rpos && h.mpos <= h.rpos + 500000) q = h.mpos;
		if(q > bd->rpos) bd->rpos = q;
		if(bd->tid == -1) bd->tid = in->tid;
		if(bd->hits.size() <= 1) bd->strand = h.strand;
		// add_intervals (:106-158): only BAM_CMATCH adds coverage; extract_splices (rnacore/hit.cc:77-104)
		chain_t spl;
		p = h.pos;
		for(int k = 0; k < nc; k++)
		{
			uint32_t op = cig[k] & 0xf, len = cig[k] >> 4;
			if((0x3C1A7 >> (op << 1)) & 2) p += (int32_t)len;
			if(op == 0) bd->mmap.add(p - (int32_t)len, p, 1);
			if(op == 3 && k != 0 && k != nc - 1) { spl.push_back(p - (int32_t)len); spl.push_back(p); }
		}
		if(!spl.empty()) bd->hcst.add(spl, (int)bd->hits.size() - 1, h.xs);
	}
	bd->splices = bd->hcst.get_splices();
	// bundle_base::compute_strand (:205-225)
	if(prm->library_type == 0)
	{
		int np = 0, nq = 0;
		for(size_t i = 0; i < bd->hits.size(); i++) { if(bd->hits[i].xs == '+') np++; if(bd->hits[i].xs == '-') nq++; }
		bd->strand = np > nq ? '+' : (np < nq ? '-' : '.');
	}
	return bd;
}

void orc_bundle_free(void *b) { delete (bundle*)b; }

int orc_bundle_evidence(void *b, void *bagp)
{
	bundle &bd = *(bundle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	std::vector<int32_t> &x = bag.ints("bundle");
	x.clear();
	x.push_back(bd.lpos); x.push_back(bd.rpos); x.push_back((int32_t)bd.strand); x.push_back((int32_t)bd.hits.size());
	bag.ints("hits").assign(bd.input_index.begin(), bd.input_index.end());
	dump_segments(bd.mmap, bag, "seg");
	bag.ints("splices") = bd.splices;
	dump_chain_set(bd.hcst, bag, "hcst", (int)bd.hits.size(), "hit_chain");
	return 0;
}

int orc_bundle_fragments(void *b, void *bagp)
{
	bundle &bd = *(bundle*)b;
	build_fragments(bd);
	dump_frgs(bd, *(orc_bag*)bagp, "frgs");
	return 0;
}

int orc_bundle_graph(void *b, void *bagp)
{
	bundle &bd = *(bundle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	graph gr;
	builder_out bo;
	build_graph(bd, gr, bo);
	dump_builder(bo, bag, "");
	dump_graph(gr, bag, "");
	return bo.repeated_bounds ? -1 : 0;            // where the reference asserts
}

// bundle::bridge (meta/bundle.cc:55-88)
int orc_bundle_bridge(void *b, void *bagp)
{
	bundle &bd = *(bundle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	graph gr;
	builder_out bo;
	build_graph(bd, gr, bo);
	if(bo.repeated_bounds) return -1;                 // where the reference asserts (see builder_out)
	dump_builder(bo, bag, "");
	dump_graph(gr, bag, "");
	return cluster_solve_update(gr, bd, bd.prm, bag, "", false);
}

// bundle_base::build_phase_set against the bundle's own splice graph (transform(bd, gr, false))
int orc_bundle_phase(void *b, void *bagp)
{
	bundle &bd = *(bundle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	graph gr;
	builder_out bo;
	build_graph(bd, gr, bo);
	if(bo.repeated_bounds) return -1;                 // where the reference asserts (see builder_out)
	std::map<chain_t, int> ps;
	build_phase_set(bd, gr, ps);
	std::vector<int32_t> &po = bag.ints("phase_off");
	std::vector<int32_t> &pv = bag.ints("phase_val");
	std::vector<int32_t> &pc = bag.ints("phase_cnt");
	po.clear(); pv.clear(); pc.clear();
	po.push_back(0);
	for(std::map<chain_t, int>::const_iterator it = ps.begin(); it != ps.end(); it++)
	{
		pv.insert(pv.end(), it->first.begin(), it->first.end());
		po.push_back((int32_t)pv.size());
		pc.push_back(it->second);
	}
	return (int)pc.size();
}

// identify_boundaries + remove_false_boundaries on the bundle's own splice graph, bundle in its current state
int orc_bundle_revise(void *b, void *bagp)
{
	bundle &bd = *(bundle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	graph gr;
	builder_out bo;
	build_graph(bd, gr, bo);
	if(bo.repeated_bounds) return -1;                 // where the reference asserts (see builder_out)
	revision rv;
	revise_graph(bd, gr, rv);
	std::vector<int32_t> &re = bag.ints("rev_edge");
	std::vector<double> &rw = bag.reals("rev_edge_d");
	std::vector<int32_t> &ge = bag.ints("rev_graph_edge");
	std::vector<double> &gw = bag.reals("rev_graph_edge_d");
	std::vector<int32_t> &vc = bag.ints("rev_vert");
	std::vector<double> &vr = bag.reals("rev_vert_d");
	re.clear(); rw.clear(); ge.clear(); gw.clear(); vc.clear(); vr.clear();
	for(size_t i = 0; i < rv.added.size(); i++) { re.push_back(rv.added[i][0]); re.push_back(rv.added[i][1]); rw.push_back(rv.added_w[i]); }
	for(int i = 0; i < gr.nv(); i++)
	{
		for(auto &pr : gr.out[i]) { ge.push_back(i); ge.push_back(pr.first); gw.push_back(gr.edges[pr.second].w); }
		vc.push_back(rv.leave_cnt[i]); vc.push_back(rv.come_cnt[i]);
		vr.push_back(rv.leave_ratio[i]); vr.push_back(rv.come_ratio[i]);
	}
	return (int)rw.size();
}

int orc_bundle_set_sample(void *b, int sample_id)
{
	((bundle*)b)->sample = sample_id;
	return 0;
}

static void dump_support(const graph &gr, const support &s, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &se = bag.ints(pre + "sup_edge"), &so = bag.ints(pre + "sup_off"), &ss = bag.ints(pre + "sup_sample");
	std::vector<int32_t> &to = bag.ints(pre + "sup_set_off"), &ts = bag.ints(pre + "sup_set");
	std::vector<double> &sa = bag.reals(pre + "sup_abd"), &sb = bag.reals(pre + "sup_sabd"), &sl = bag.reals(pre + "sup_loss");
	se.clear(); so.clear(); ss.clear(); to.clear(); ts.clear(); sa.clear(); sb.clear(); sl.clear();
	so.push_back(0); to.push_back(0);
	for(int i = 0; i < gr.nv(); i++)
	{
		for(int x = 0; x < 4; x++) sl.push_back(s.loss[i][x]);
		for(auto &pr : gr.out[i])
		{
			const int e = pr.second;
			se.push_back(i); se.push_back(pr.first); se.push_back(s.count[e]);
			sa.push_back(s.abd[e]);
			for(auto &z : s.spabd[e]) { ss.push_back(z.first); sb.push_back(z.second); }
			so.push_back((int32_t)ss.size());
			ts.insert(ts.end(), s.samples[e].begin(), s.samples[e].end());
			to.push_back((int32_t)ts.size());
		}
	}
}

// the cross-sample support features of assembler::assemble(vector<bundle*>) (meta/assembler.cc:177-373)
int orc_group_support(void **bs, int n, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	if(n < 2) return -1;
	std::vector<graph> grs;
	std::vector<support> sups;
	graph gx;
	support sx;
	if(group_support((bundle**)bs, n, grs, sups, gx, sx)) return -1;
	for(int k = 0; k < n; k++)
	{
		char pre[32];
		snprintf(pre, sizeof(pre), "m%d_", k);
		dump_support(grs[k], sups[k], bag, pre);
	}
	dump_support(gx, sx, bag, "x_");
	return 0;
}

// assembler::bridge (meta/assembler.cc:977-1018) with combine_bundles (:152-175) and bundle::combine (meta/bundle.cc:90-107)
int orc_group_bridge(void **bs, int n, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	if(n < 2) return -1;
	bundle &b0 = *(bundle*)bs[0];
	bundle cb;
	cb.prm = b0.prm;
	cb.tid = b0.tid; cb.lpos = b0.lpos; cb.rpos = b0.rpos; cb.strand = b0.strand;
	std::vector<std::pair<int, int> > v;
	for(int k = 0; k < n; k++) v.push_back(std::make_pair(k, (int)((bundle*)bs[k])->mmap.segments().size()));
	std::sort(v.begin(), v.end(), [](const std::pair<int, int> &x, const std::pair<int, int> &y) { return x.second > y.second; });
	std::vector<int32_t> &ord = bag.ints("combine_order");
	ord.clear();
	for(size_t i = 0; i < v.size(); i++)
	{
		const bundle &bb = *(bundle*)bs[v[i].first];
		if(cb.lpos > bb.lpos) cb.lpos = bb.lpos;
		if(cb.rpos < bb.rpos) cb.rpos = bb.rpos;
		cb.hcst.add(bb.hcst);
		cb.fcst.add(bb.fcst);
		cb.mmap.add(bb.mmap);
		ord.push_back(v[i].first);
	}
	dump_chain_set(cb.hcst, bag, "cb_hcst", 0, "cb_hit_chain");
	dump_chain_set(cb.fcst, bag, "cb_fcst", 0, "cb_frg_chain");
	dump_segments(cb.mmap, bag, "cb_seg");
	std::vector<int32_t> &cbb = bag.ints("cb_bundle");
	cbb.clear();
	cbb.push_back(cb.lpos); cbb.push_back(cb.rpos); cbb.push_back((int32_t)cb.strand);
	graph gr;
	builder_out bo;
	build_graph(cb, gr, bo);
	if(bo.repeated_bounds) return -1;                 // where the reference asserts (see builder_out)
	dump_builder(bo, bag, "cb_");
	dump_graph(gr, bag, "cb_");
	int total = 0;
	for(int k = 0; k < n; k++)
	{
		char pre[32];
		snprintf(pre, sizeof(pre), "b%d_", k);
		total += cluster_solve_update(gr, *(bundle*)bs[k], b0.prm, bag, pre, true);
	}
	return total;
}

namespace {

// bundle_group::resolve (meta/bundle_group.cc:26-56) on n sorted splice lists
int resolve_lists(const std::vector<const std::vector<int32_t>*> &sp, const orc_params *prm, orc_bag &bag)
{
	const int n = (int)sp.size();
	// build_splice_index (:150-172)
	std::map<int32_t, std::set<int> > sindex;
	for(int k = 0; k < n; k++) for(size_t i = 0; i < sp[k]->size(); i++) sindex[(*sp[k])[i]].insert(k);
	// disjoint sets with a size slot at the representative (rnacore/disjoint_set.h; union by rank, boost::disjoint_sets)
	std::vector<int> parent(n), rank(n, 0), size(n, 1);
	for(int k = 0; k < n; k++) parent[k] = k;
	struct { std::vector<int> *p; int find(int x) { int r = x; while((*p)[r] != r) r = (*p)[r]; while((*p)[x] != r) { int nx = (*p)[x]; (*p)[x] = r; x = nx; } return r; } } ds;
	ds.p = &parent;
	std::vector<bool> grouped(n, false);
	double thr[2] = {prm->max_grouping_similarity, prm->min_grouping_similarity};
	for(int round = 0; round < 2; round++)
	{
		for(std::map<int32_t, std::set<int> >::iterator z = sindex.begin(); z != sindex.end(); ++z)
		{
			if(z->second.size() <= 1) continue;
			// filter (:344-358)
			std::vector<int> ss;
			for(std::set<int>::iterator it = z->second.begin(); it != z->second.end(); ++it)
			{
				if(grouped[*it]) continue;
				if(size[ds.find(*it)] >= prm->max_group_size) { grouped[*it] = true; continue; }
				ss.push_back(*it);
			}
			// build_splice_similarity (:190-231)
			typedef std::pair<std::pair<int, int>, double> PPID;
			std::vector<PPID> vpid;
			for(size_t xi = 0; xi < ss.size(); xi++)
			{
				int i = ss[xi];
				if(sp[i]->size() / 2.0 > prm->max_num_junctions_to_combine) continue;
				int pi = ds.find(i);
				for(size_t xj = 0; xj < ss.size(); xj++)
				{
					int j = ss[xj];
					if(i >= j) continue;
					if(sp[j]->size() / 2.0 > prm->max_num_junctions_to_combine) continue;
					if(pi == ds.find(j)) continue;
					std::vector<int32_t> vv(sp[i]->size() + sp[j]->size(), 0);
					int c = (int)(std::set_intersection(sp[i]->begin(), sp[i]->end(), sp[j]->begin(), sp[j]->end(), vv.begin()) - vv.begin());
					int small = (int)std::min(sp[i]->size(), sp[j]->size());
					double r = c * 1.0 / small;
					if(c <= 0.50) continue;
					if(r < thr[round]) continue;
					vpid.push_back(PPID(std::make_pair(i, j), r));
				}
			}
			std::sort(vpid.begin(), vpid.end(), [](const PPID &x, const PPID &y) { return x.second > y.second; });
			// augment_disjoint_set (:296-318)
			for(size_t k = 0; k < vpid.size(); k++)
			{
				int px = ds.find(vpid[k].first.first), py = ds.find(vpid[k].first.second);
				if(px == py) continue;
				int sx = size[px], sy = size[py];
				if(sx >= prm->max_group_size || sy >= prm->max_group_size) continue;
				if(rank[px] > rank[py]) parent[py] = px;
				else { parent[px] = py; if(rank[px] == rank[py]) rank[py]++; }
				size[ds.find(px)] = sx + sy;
			}
		}
	}
	// build_groups (:320-342)
	std::map<int, int> mm;
	std::vector<std::vector<int> > gvv;
	for(int i = 0; i < n; i++)
	{
		int p = ds.find(i);
		if(mm.find(p) == mm.end()) { mm[p] = (int)gvv.size(); gvv.push_back(std::vector<int>(1, i)); }
		else gvv[mm[p]].push_back(i);
	}
	std::vector<int32_t> &off = bag.ints("gvv_off"), &val = bag.ints("gvv_val");
	off.assign(1, 0); val.clear();
	for(size_t i = 0; i < gvv.size(); i++) { val.insert(val.end(), gvv[i].begin(), gvv[i].end()); off.push_back((int32_t)val.size()); }
	return 0;
}

} // namespace

// bundle_group::resolve on the bundles' splice lists
int orc_group_resolve(void **bs, int n, const orc_params *prm, void *bagp)
{
	std::vector<const std::vector<int32_t>*> sp(n);
	for(int k = 0; k < n; k++) sp[k] = &((bundle*)bs[k])->splices;
	return resolve_lists(sp, prm, *(orc_bag*)bagp);
}

// the same on given lists: list k is list_val[list_off[k] .. list_off[k + 1])
int orc_group_resolve_lists(int n, const int64_t *list_off, const int32_t *list_val, const orc_params *prm, void *bagp)
{
	std::vector<std::vector<int32_t> > lists(n);
	std::vector<const std::vector<int32_t>*> sp(n);
	for(int k = 0; k < n; k++)
	{
		lists[k].assign(list_val + list_off[k], list_val + list_off[k + 1]);
		sp[k] = &lists[k];
	}
	return resolve_lists(sp, prm, *(orc_bag*)bagp);
}


// the permutation libstdc++'s std::sort leaves for the comparator key[a] < key[b] (a partial order when keys tie)
int orc_std_sort_perm(const int32_t *keys, int32_t n, int32_t *perm)
{
	std::vector<int32_t> v(n);
	for(int i = 0; i < n; i++) v[i] = i;
	std::sort(v.begin(), v.end(), [keys](int32_t a, int32_t b) { return keys[a] < keys[b]; });
	for(int i = 0; i < n; i++) perm[i] = v[i];
	return 0;
}

}
