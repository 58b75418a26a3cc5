// TEST INFRASTRUCTURE ONLY (oracle/): drives the reference's OWN classes (compiled unchanged
// from /root/reference, see oracle/Makefile) through the hot path and dumps what they computed
// as flat named arrays (orc_api.h).  This file contains no algorithm of its own: it only calls
// the reference in the order the reference's callers do and copies fields out.
//
// Call orders mirrored:
//   ref_bundle_new       meta/generator.cc:155-179 (add_hit_intervals per hit) + :203-227 (generate)
//   ref_bundle_fragments meta/assembler.cc:39       (build_fragments)
//   ref_bundle_graph     meta/assembler.cc:930-934  (graph_builder::build + build_vertex_index)
//   ref_bundle_bridge    meta/bundle.cc:55-88       (bundle::bridge)
//   ref_group_bridge     meta/assembler.cc:977-1018 (assembler::bridge)
//   ref_group_resolve    meta/bundle_group.cc:26-56 (bundle_group::resolve)
#include "orc_api.h"
#include "orc_bag.h"
#include "compat/hts_shim.h"

#include "bundle.h"
#include "bundle_group.h"
#include "generator.h"
#include "previewer.h"
#include "assembler.h"
#include "../integration/adapter.h"
#include "graph_builder.h"
#include "graph_cluster.h"
#include "graph_reviser.h"
#include "bridge_solver.h"
#include "essential.h"
#include "parameters.h"
#include "phase_set.h"
#include "sample_profile.h"

#include <atomic>
#include <chrono>
#include <cmath>
#include <thread>
#include <set>
#include <unordered_map>
#include <mutex>
#include <string>
#include <vector>

namespace {

struct ref_handle
{
	parameters cfg;
	sample_profile sp;
	bundle bd;
	std::vector<int> keep;        // input index of every stored hit
	ref_handle() : sp(0, 1000000), bd(cfg, sp) {}
};

void apply_params(const orc_params *p, parameters &cfg, sample_profile &sp)
{
	cfg.verbose = 0;
	cfg.min_junction_support = p->min_junction_support;
	cfg.normal_junction_threshold = p->normal_junction_threshold;
	cfg.extend_junction_threshold = p->extend_junction_threshold;
	cfg.min_subregion_gap = p->min_subregion_gap;
	cfg.min_subregion_length = p->min_subregion_length;
	cfg.min_subregion_overlap = p->min_subregion_overlap;
	cfg.min_guaranteed_edge_weight = p->min_guaranteed_edge_weight;
	cfg.max_reads_partition_gap = p->max_reads_partition_gap;
	cfg.bridge_end_relaxing = p->bridge_end_relaxing;
	cfg.bridge_dp_solution_size = p->bridge_dp_solution_size;
	cfg.bridge_dp_stack_size = p->bridge_dp_stack_size;
	cfg.max_group_size = p->max_group_size;
	cfg.max_num_junctions_to_combine = p->max_num_junctions_to_combine;
	cfg.min_grouping_similarity = p->min_grouping_similarity;
	cfg.max_grouping_similarity = p->max_grouping_similarity;
	cfg.min_boundary_log_ratio = p->min_boundary_log_ratio;
	cfg.max_group_boundary_distance = p->max_group_boundary_distance;
	sp.library_type = p->library_type;
	sp.insertsize_low = p->insertsize_low;
	sp.insertsize_high = p->insertsize_high;
}

std::string qname_of(uint64_t q)
{
	char buf[32];
	snprintf(buf, sizeof(buf), "q%016llx", (unsigned long long)q);
	return std::string(buf);
}

void dump_chain_set(const chain_set &cs, orc_bag &bag, const std::string &pre, int nh, const std::string &hname)
{
	std::vector<int32_t> &off = bag.ints(pre + "_off");
	std::vector<int32_t> &val = bag.ints(pre + "_val");
	std::vector<int32_t> &cnt = bag.ints(pre + "_cnt");
	std::vector<int32_t> &grp = bag.ints(pre + "_grp");
	off.clear(); val.clear(); cnt.clear(); grp.clear();
	std::vector< std::vector<int> > flat(cs.chains.size());
	off.push_back(0);
	int c = 0;
	for(size_t i = 0; i < cs.chains.size(); i++)
	{
		for(size_t j = 0; j < cs.chains[i].size(); j++)
		{
			const PVI3 &p = cs.chains[i][j];
			val.insert(val.end(), p.first.begin(), p.first.end());
			off.push_back((int32_t)val.size());
			cnt.push_back(p.second[0]);
			cnt.push_back(p.second[1]);
			cnt.push_back(p.second[2]);
			grp.push_back((int32_t)i);
			flat[i].push_back(c++);
		}
	}
	std::vector<int32_t> &hc = bag.ints(hname);
	std::vector<int32_t> &hx = bag.ints(hname + "_xs");
	hc.assign(nh, -1);
	hx.assign(nh, -1);
	for(std::map<int, AI3>::const_iterator it = cs.hmap.begin(); it != cs.hmap.end(); ++it)
	{
		if(it->first < 0 || it->first >= nh) continue;
		hc[it->first] = flat[it->second[0]][it->second[1]];
		hx[it->first] = it->second[2];
	}
}

void dump_segments(const split_interval_map &m, orc_bag &bag, const std::string &name)
{
	std::vector<int32_t> &seg = bag.ints(name);
	seg.clear();
	for(SIMI it = m.begin(); it != m.end(); ++it)
	{
		seg.push_back(lower(it->first));
		seg.push_back(upper(it->first));
		seg.push_back(it->second);
	}
}

void dump_evidence(ref_handle &h, orc_bag &bag)
{
	bundle &bd = h.bd;
	std::vector<int32_t> &b = bag.ints("bundle");
	b.clear();
	b.push_back(bd.lpos);
	b.push_back(bd.rpos);
	b.push_back((int32_t)bd.strand);
	b.push_back((int32_t)bd.hits.size());
	std::vector<int32_t> &kp = bag.ints("hits");
	kp.assign(h.keep.begin(), h.keep.end());
	dump_segments(bd.mmap, bag, "seg");
	bag.ints("splices") = bd.splices;
	dump_chain_set(bd.hcst, bag, "hcst", (int)bd.hits.size(), "hit_chain");
}

void dump_frgs(bundle_base &bd, orc_bag &bag, const std::string &name)
{
	std::vector<int32_t> &f = bag.ints(name);
	f.clear();
	for(size_t i = 0; i < bd.frgs.size(); i++)
	{
		f.push_back(bd.frgs[i][0]);
		f.push_back(bd.frgs[i][1]);
		f.push_back(bd.frgs[i][2]);
	}
}

// returns, per partial exon, whether it is one of the 1-bp stubs whose `max` the reference never sets
std::vector<char> dump_builder(graph_builder &gb, parameters &cfg, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &jc = bag.ints(pre + "junc");
	jc.clear();
	for(size_t i = 0; i < gb.junctions.size(); i++)
	{
		const junction &j = gb.junctions[i];
		jc.push_back(j.lpos); jc.push_back(j.rpos); jc.push_back(j.count);
		jc.push_back(j.xs0); jc.push_back(j.xs1); jc.push_back(j.xs2);
		jc.push_back((int32_t)j.strand); jc.push_back(j.lexon); jc.push_back(j.rexon);
	}
	std::vector<int32_t> &pe = bag.ints(pre + "pexon");
	std::vector<double> &pd = bag.reals(pre + "pexon_d");
	pe.clear(); pd.clear();
	std::vector<char> stubs(gb.pexons.size(), 0);
	for(size_t i = 0; i < gb.pexons.size(); i++)
	{
		const partial_exon &p = gb.pexons[i];
		pe.push_back(p.lpos); pe.push_back(p.rpos); pe.push_back(p.ltype); pe.push_back(p.rtype);
		pe.push_back(gb.regional[i] ? 1 : 0);
		// partial_exon::max is left uninitialised for the 1-bp stub pexons
		// (rnacore/region.cc:118-121, :135-138, :162-165): report -1 there
		bool stub = (p.rpos - p.lpos == 1 && p.ave == cfg.min_guaranteed_edge_weight && p.dev == 1.0);
		stubs[i] = stub ? 1 : 0;
		pd.push_back(p.ave); pd.push_back(p.dev); pd.push_back(stub ? -1.0 : p.max); pd.push_back(p.pvalue);
	}
	return stubs;
}

// vertex i (inner) is partial exon i - 1 (rnacore/graph_builder.cc:305-341): its maxcov is unset exactly when the pexon's max is
void dump_graph(splice_graph &gr, parameters &cfg, orc_bag &bag, const std::string &pre, const std::vector<char> &stubs)
{
	std::vector<int32_t> &vi = bag.ints(pre + "vert");
	std::vector<double> &vd = bag.reals(pre + "vert_d");
	std::vector<int32_t> &ei = bag.ints(pre + "edge");
	std::vector<double> &ed = bag.reals(pre + "edge_d");
	vi.clear(); vd.clear(); ei.clear(); ed.clear();
	int n = (int)gr.num_vertices();
	for(int i = 0; i < n; i++)
	{
		const vertex_info &v = gr.get_vertex_info(i);
		double w = gr.get_vertex_weight(i);
		vi.push_back(v.lpos); vi.push_back(v.rpos); vi.push_back(v.length); vi.push_back(v.type);
		vi.push_back(v.regional ? 1 : 0);
		bool stub = (i != 0 && i != n - 1 && (size_t)(i - 1) < stubs.size() && stubs[i - 1]);
		vd.push_back(w); vd.push_back(v.stddev); vd.push_back(stub ? -1.0 : v.maxcov);
	}
	for(int i = 0; i < n; i++)
	{
		PEEI pe = gr.out_edges(i);
		for(edge_iterator it = pe.first; it != pe.second; ++it)
		{
			edge_descriptor e = *it;
			ei.push_back(e->source()); ei.push_back(e->target()); ei.push_back(gr.get_edge_info(e).strand);
			ed.push_back(gr.get_edge_weight(e));
		}
	}
	std::vector<int32_t> &gs = bag.ints(pre + "graph");
	gs.clear();
	gs.push_back((int32_t)gr.strand);
}

void dump_clusters(const std::vector<pereads_cluster> &vc, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &bo = bag.ints(pre + "clu_bounds");
	std::vector<int32_t> &ex = bag.ints(pre + "clu_extend");
	std::vector<int32_t> &ct = bag.ints(pre + "clu_count");
	std::vector<int32_t> &o1 = bag.ints(pre + "clu_c1_off");
	std::vector<int32_t> &v1 = bag.ints(pre + "clu_c1_val");
	std::vector<int32_t> &o2 = bag.ints(pre + "clu_c2_off");
	std::vector<int32_t> &v2 = bag.ints(pre + "clu_c2_val");
	std::vector<int32_t> &of = bag.ints(pre + "clu_fr_off");
	std::vector<int32_t> &vf = bag.ints(pre + "clu_fr_val");
	bo.clear(); ex.clear(); ct.clear(); o1.clear(); v1.clear(); o2.clear(); v2.clear(); of.clear(); vf.clear();
	o1.push_back(0); o2.push_back(0); of.push_back(0);
	for(size_t i = 0; i < vc.size(); i++)
	{
		const pereads_cluster &pc = vc[i];
		bo.insert(bo.end(), pc.bounds.begin(), pc.bounds.end());
		ex.insert(ex.end(), pc.extend.begin(), pc.extend.end());
		ct.push_back(pc.count);
		v1.insert(v1.end(), pc.chain1.begin(), pc.chain1.end());
		o1.push_back((int32_t)v1.size());
		v2.insert(v2.end(), pc.chain2.begin(), pc.chain2.end());
		o2.push_back((int32_t)v2.size());
		vf.insert(vf.end(), pc.frlist.begin(), pc.frlist.end());
		of.push_back((int32_t)vf.size());
	}
}

void dump_opt(const std::vector<bridge_path> &opt, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &o = bag.ints(pre + "opt");
	std::vector<double> &os = bag.reals(pre + "opt_score");
	std::vector<int32_t> &co = bag.ints(pre + "opt_chain_off");
	std::vector<int32_t> &cv = bag.ints(pre + "opt_chain_val");
	std::vector<int32_t> &wo = bag.ints(pre + "opt_whole_off");
	std::vector<int32_t> &wv = bag.ints(pre + "opt_whole_val");
	o.clear(); os.clear(); co.clear(); cv.clear(); wo.clear(); wv.clear();
	co.push_back(0); wo.push_back(0);
	for(size_t i = 0; i < opt.size(); i++)
	{
		const bridge_path &p = opt[i];
		o.push_back(p.type); o.push_back(p.strand); o.push_back(p.choices);
		os.push_back(p.score);
		cv.insert(cv.end(), p.chain.begin(), p.chain.end());
		co.push_back((int32_t)cv.size());
		wv.insert(wv.end(), p.whole.begin(), p.whole.end());
		wo.push_back((int32_t)wv.size());
	}
}

// meta/bundle.cc:66-79 / meta/assembler.cc:989-1012: cluster, solve, update one bundle against gr
int cluster_solve_update(splice_graph &gr, bundle &bd, const parameters &cfg, orc_bag &bag, const std::string &pre, bool skip_if_empty)
{
	std::vector<pereads_cluster> vc;
	graph_cluster gc(gr, bd, cfg.max_reads_partition_gap, false);
	gc.build_pereads_clusters(vc);
	dump_frgs(bd, bag, pre + "frgs_clustered");
	dump_clusters(vc, bag, pre);
	int cnt = 0;
	if(skip_if_empty && vc.size() <= 0)
	{
		dump_opt(std::vector<bridge_path>(), bag, pre);
	}
	else
	{
		bridge_solver bs(gr, vc, cfg, bd.sp.insertsize_low, bd.sp.insertsize_high);
		dump_opt(bs.opt, bag, pre);
		for(size_t k = 0; k < vc.size(); k++)
		{
			if(bs.opt[k].type <= 0) continue;
			cnt += bd.update_bridges(vc[k].frlist, bs.opt[k].chain, bs.opt[k].strand);
		}
	}
	dump_frgs(bd, bag, pre + "frgs");
	dump_chain_set(bd.fcst, bag, pre + "fcst", (int)bd.frgs.size(), pre + "frg_chain");
	dump_segments(bd.mmap, bag, pre + "seg");
	std::vector<int32_t> &bc = bag.ints(pre + "bridged");
	bc.clear();
	bc.push_back(cnt);
	return cnt;
}

} // namespace

extern "C" {

void *ref_bundle_new(const orc_bundle_in *in, const orc_params *prm)
{
	ref_handle *h = new ref_handle;
	apply_params(prm, h->cfg, h->sp);
	bundle_base &bb = h->bd;
	bam1_t b1t;
	for(int i = 0; i < in->n_hits; i++)
	{
		uint32_t c0 = in->cigar_off[i];
		uint32_t c1 = in->cigar_off[i + 1];
		hts_shim_record rec = hts_shim_make_record(in->tid, in->pos[i], 60, in->flag[i], in->tid, in->mpos[i], in->isize[i],
				qname_of(in->qid[i]), in->cigar + c0, c1 - c0, (char)in->xs[i], '.', 1, 1, -1);
		hts_shim_view(rec, &b1t);
		hit ht(&b1t, i);
		ht.set_tags(&b1t);
		ht.strand = (char)in->strand[i];
		size_t before = bb.hits.size();
		bb.add_hit_intervals(ht, &b1t);
		if(bb.hits.size() > before) h->keep.push_back(i);
	}
	// meta/generator.cc:203-227
	bb.add_buf_intervals();
	bb.splices = bb.hcst.get_splices();
	h->bd.chrm = "chr";
	h->bd.compute_strand(h->sp.library_type);
	return h;
}

void ref_bundle_free(void *b) { delete (ref_handle*)b; }


// ---- timing entry (bench.py --impl reference, cpu_baseline): the reference's own bundle path with nothing of the checker in
// the timed region.  ref_timing_new fabricates the BAM records and constructs the `hit` objects (hit::hit + set_tags + the
// generator's strand fix-up) BEFORE any clock starts -- the GPU arm starts from packed hits too.  ref_timing_run then does, per
// bundle and on a pool of `threads` workers (one bundle per task, the granularity of aletsch -t N, meta/incubator.cc:615-635):
// add_hit_intervals per hit + the end of generator::generate (meta/generator.cc:203-227) + build_fragments + the reference's
// own bundle::bridge() (meta/bundle.cc:55-88), on a fresh bundle object, and returns the wall time of the pool.
struct ref_timing_bundle
{
	std::vector<hts_shim_record> recs;
	std::vector<hit> hits;
};
struct ref_timing
{
	parameters cfg;
	sample_profile sp;
	std::vector<ref_timing_bundle> bundles;
	ref_timing() : sp(0, 1000000) {}
};

void *ref_timing_new(int n_bundles, const orc_bundle_in *ins, const orc_params *prm)
{
	ref_timing *t = new ref_timing;
	apply_params(prm, t->cfg, t->sp);
	t->bundles.resize(n_bundles);
	for(int k = 0; k < n_bundles; k++)
	{
		const orc_bundle_in *in = ins + k;
		ref_timing_bundle &tb = t->bundles[k];
		tb.recs.reserve(in->n_hits);
		tb.hits.reserve(in->n_hits);
		for(int i = 0; i < in->n_hits; i++)
		{
			uint32_t c0 = in->cigar_off[i], c1 = in->cigar_off[i + 1];
			tb.recs.push_back(hts_shim_make_record(in->tid, in->pos[i], 60, in->flag[i], in->tid, in->mpos[i], in->isize[i],
					qname_of(in->qid[i]), in->cigar + c0, c1 - c0, (char)in->xs[i], '.', 1, 1, -1));
		}
		for(int i = 0; i < in->n_hits; i++)
		{
			bam1_t b1t;
			hts_shim_view(tb.recs[i], &b1t);
			hit ht(&b1t, i);
			ht.set_tags(&b1t);
			ht.strand = (char)in->strand[i];
			tb.hits.push_back(ht);
		}
	}
	return t;
}

void ref_timing_free(void *t) { delete (ref_timing*)t; }

int64_t ref_timing_hits(void *tp)
{
	ref_timing *t = (ref_timing*)tp;
	int64_t n = 0;
	for(size_t k = 0; k < t->bundles.size(); k++) n += (int64_t)t->bundles[k].hits.size();
	return n;
}

// one pass over all bundles; per_bundle_bridged (may be NULL) receives the number of bridged fragments of every bundle
// (frgs of type 1 / 2 after bundle::bridge, i.e. the sum of the update_bridges return values)
int ref_timing_run(void *tp, int threads, double *seconds, int64_t *bridged, int32_t *per_bundle_bridged)
{
	ref_timing *t = (ref_timing*)tp;
	const int n = (int)t->bundles.size();
	if(threads < 1) threads = 1;
	std::atomic<int> next(0);
	std::atomic<long long> total(0);
	auto work = [&]()
	{
		while(true)
		{
			int k = next.fetch_add(1);
			if(k >= n) return;
			ref_timing_bundle &tb = t->bundles[k];
			bundle bd(t->cfg, t->sp);
			bam1_t b1t;
			for(size_t i = 0; i < tb.hits.size(); i++)
			{
				hts_shim_view(tb.recs[i], &b1t);
				bd.add_hit_intervals(tb.hits[i], &b1t);
			}
			bd.add_buf_intervals();
			bd.splices = bd.hcst.get_splices();
			bd.chrm = "chr";
			bd.compute_strand(t->sp.library_type);
			bd.build_fragments();
			bd.bridge();
			int cnt = 0;
			for(size_t f = 0; f < bd.frgs.size(); f++) if(bd.frgs[f][2] == 1 || bd.frgs[f][2] == 2) cnt++;
			if(per_bundle_bridged) per_bundle_bridged[k] = cnt;
			total += cnt;
		}
	};
	auto t0 = std::chrono::steady_clock::now();
	std::vector<std::thread> pool;
	for(int i = 0; i < threads; i++) pool.push_back(std::thread(work));
	for(size_t i = 0; i < pool.size(); i++) pool[i].join();
	auto t1 = std::chrono::steady_clock::now();
	if(seconds) *seconds = std::chrono::duration<double>(t1 - t0).count();
	if(bridged) *bridged = total.load();
	return 0;
}

// Full-size cross-check (untimed): the same per-bundle work as ref_timing_run, then three order-sensitive 64-bit digests of what
// bundle::bridge leaves behind -- digest[3k] over the mmap segments (lower, upper, coverage), [3k + 1] over frgs (h1, h2, type),
// [3k + 2] over bundle::splices -- each the wrapping sum over the rows j of row_digest(a, b, c, j).  bench.py forms the same
// digests from the views of agpu_batch_results (bench.py: view_digests).
static inline uint64_t row_digest(int32_t a, int32_t b, int32_t c, uint64_t j)
{
	uint64_t x = (uint64_t)(uint32_t)a * 0x9E3779B97F4A7C15ULL ^ (uint64_t)(uint32_t)b * 0xC2B2AE3D27D4EB4FULL
		^ (uint64_t)(uint32_t)c * 0x165667B19E3779F9ULL ^ j * 0xD6E8FEB86659FD93ULL;
	x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ULL; x ^= x >> 27; x *= 0x94D049BB133111EBULL; x ^= x >> 31;
	return x;
}
int ref_timing_digest(void *tp, int threads, uint64_t *digest)
{
	ref_timing *t = (ref_timing*)tp;
	const int n = (int)t->bundles.size();
	if(threads < 1) threads = 1;
	std::atomic<int> next(0);
	auto work = [&]()
	{
		while(true)
		{
			int k = next.fetch_add(1);
			if(k >= n) return;
			ref_timing_bundle &tb = t->bundles[k];
			bundle bd(t->cfg, t->sp);
			bam1_t b1t;
			for(size_t i = 0; i < tb.hits.size(); i++)
			{
				hts_shim_view(tb.recs[i], &b1t);
				bd.add_hit_intervals(tb.hits[i], &b1t);
			}
			bd.add_buf_intervals();
			bd.splices = bd.hcst.get_splices();
			bd.chrm = "chr";
			bd.compute_strand(t->sp.library_type);
			bd.build_fragments();
			bd.bridge();
			uint64_t d0 = 0, d1 = 0, d2 = 0, j = 0;
			for(SIMI it = bd.mmap.begin(); it != bd.mmap.end(); ++it, ++j) d0 += row_digest(lower(it->first), upper(it->first), it->second, j);
			for(size_t f = 0; f < bd.frgs.size(); f++) d1 += row_digest(bd.frgs[f][0], bd.frgs[f][1], bd.frgs[f][2], (uint64_t)f);
			for(size_t s = 0; s < bd.splices.size(); s++) d2 += row_digest(bd.splices[s], 0, 0, (uint64_t)s);
			digest[3 * (size_t)k] = d0; digest[3 * (size_t)k + 1] = d1; digest[3 * (size_t)k + 2] = d2;
		}
	};
	std::vector<std::thread> pool;
	for(int i = 0; i < threads; i++) pool.push_back(std::thread(work));
	for(size_t i = 0; i < pool.size(); i++) pool[i].join();
	return 0;
}

int ref_bundle_evidence(void *b, void *bag)
{
	dump_evidence(*(ref_handle*)b, *(orc_bag*)bag);
	return 0;
}

int ref_bundle_fragments(void *b, void *bag)
{
	ref_handle *h = (ref_handle*)b;
	h->bd.build_fragments();
	dump_frgs(h->bd, *(orc_bag*)bag, "frgs");
	return 0;
}

int ref_bundle_graph(void *b, void *bagp)
{
	ref_handle *h = (ref_handle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	splice_graph gr;
	graph_builder gb(h->bd, h->cfg, h->sp);
	gb.build(gr);
	gr.build_vertex_index();
	dump_graph(gr, h->cfg, bag, "", dump_builder(gb, h->cfg, bag, ""));
	return 0;
}

int ref_bundle_bridge(void *b, void *bagp)
{
	ref_handle *h = (ref_handle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	splice_graph gr;
	graph_builder gb(h->bd, h->cfg, h->sp);
	gb.build(gr);
	gr.build_vertex_index();
	dump_graph(gr, h->cfg, bag, "", dump_builder(gb, h->cfg, bag, ""));
	return cluster_solve_update(gr, h->bd, h->cfg, bag, "", false);
}

// bundle_base::build_phase_set (rnacore/bundle_base.cc:338-418) against the bundle's own (unrevised) splice graph, i.e. the
// graph of transform(bd, gr, false); the map is dumped in its own (lexicographic) order
int ref_bundle_phase(void *b, void *bagp)
{
	ref_handle *h = (ref_handle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	splice_graph gr;
	graph_builder gb(h->bd, h->cfg, h->sp);
	gb.build(gr);
	gr.build_vertex_index();
	phase_set ps;
	h->bd.build_phase_set(ps, gr);
	std::vector<int32_t> &po = bag.ints("phase_off");
	std::vector<int32_t> &pv = bag.ints("phase_val");
	std::vector<int32_t> &pc = bag.ints("phase_cnt");
	po.clear(); pv.clear(); pc.clear();
	po.push_back(0);
	for(MVII::const_iterator it = ps.pmap.begin(); it != ps.pmap.end(); it++)
	{
		pv.insert(pv.end(), it->first.begin(), it->first.end());
		po.push_back((int32_t)pv.size());
		pc.push_back(it->second);
	}
	return (int)pc.size();
}

// the revising half of assembler::transform(bd, gr, true) (meta/assembler.cc:930-944) on the bundle in its current state
// (call after ref_bundle_bridge, as assembler::assemble does): identify_boundaries, remove_false_boundaries,
// refine_splice_graph.  The loop of identify_boundaries is restated here around the reference's own
// identify_start_boundary / identify_end_boundary so that the order in which the edges are added can be dumped
// (rev_edge = src dst per added edge, rev_edge_d = weight); rev_graph_edge / rev_graph_edge_d is the whole revised graph in
// out-edge order, rev_vert / rev_vert_d the unbridge_* annotations of every vertex.
int ref_bundle_revise(void *b, void *bagp)
{
	ref_handle *h = (ref_handle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	splice_graph gr;
	graph_builder gb(h->bd, h->cfg, h->sp);
	gb.build(gr);
	gr.build_vertex_index();
	std::vector<int32_t> &re = bag.ints("rev_edge");
	std::vector<double> &rw = bag.reals("rev_edge_d");
	re.clear(); rw.clear();
	int n = (int)gr.num_vertices() - 1;
	std::set<std::pair<int, int> > seen;
	for(int i = 0; i <= n; i++)
	{
		PEEI pe = gr.out_edges(i);
		for(edge_iterator it = pe.first; it != pe.second; ++it) seen.insert(std::make_pair((*it)->source(), (*it)->target()));
	}
	while(true)
	{
		bool b1 = identify_start_boundary(gr, h->cfg.min_boundary_log_ratio);
		if(b1)
		{
			PEEI pe = gr.out_edges(0);
			for(edge_iterator it = pe.first; it != pe.second; ++it)
			{
				std::pair<int, int> k((*it)->source(), (*it)->target());
				if(seen.find(k) != seen.end()) continue;
				seen.insert(k);
				re.push_back(k.first); re.push_back(k.second); rw.push_back(gr.get_edge_weight(*it));
			}
		}
		bool b2 = identify_end_boundary(gr, h->cfg.min_boundary_log_ratio);
		if(b2)
		{
			PEEI pe = gr.in_edges(n);
			for(edge_iterator it = pe.first; it != pe.second; ++it)
			{
				std::pair<int, int> k((*it)->source(), (*it)->target());
				if(seen.find(k) != seen.end()) continue;
				seen.insert(k);
				re.push_back(k.first); re.push_back(k.second); rw.push_back(gr.get_edge_weight(*it));
			}
		}
		if(b1 == false && b2 == false) break;
	}
	remove_false_boundaries(gr, h->bd, h->cfg);
	refine_splice_graph(gr);
	std::vector<int32_t> &ge = bag.ints("rev_graph_edge");
	std::vector<double> &gw = bag.reals("rev_graph_edge_d");
	std::vector<int32_t> &vc = bag.ints("rev_vert");
	std::vector<double> &vr = bag.reals("rev_vert_d");
	ge.clear(); gw.clear(); vc.clear(); vr.clear();
	for(int i = 0; i <= n; i++)
	{
		PEEI pe = gr.out_edges(i);
		for(edge_iterator it = pe.first; it != pe.second; ++it)
		{
			ge.push_back((*it)->source()); ge.push_back((*it)->target());
			gw.push_back(gr.get_edge_weight(*it));
		}
		const vertex_info &vi = gr.get_vertex_info(i);
		vc.push_back(vi.unbridge_leaving_count); vc.push_back(vi.unbridge_coming_count);
		vr.push_back(vi.unbridge_leaving_ratio); vr.push_back(vi.unbridge_coming_ratio);
	}
	return (int)rw.size();
}

namespace {

// transcripts of a transcript_set, sorted by (strand, exons) so that the dump does not depend on hash order:
// trst_off / trst_exon (l r per exon), trst_meta (strand, count of samples), trst_cov (coverage)
void dump_transcripts(transcript_set &tm, orc_bag &bag)
{
	std::vector<transcript> v = tm.get_transcripts(0);
	std::sort(v.begin(), v.end(), [](const transcript &x, const transcript &y)
	{
		if(x.strand != y.strand) return x.strand < y.strand;
		if(x.exons != y.exons) return x.exons < y.exons;
		return x.coverage < y.coverage;
	});
	std::vector<int32_t> &off = bag.ints("trst_off"), &ex = bag.ints("trst_exon"), &me = bag.ints("trst_meta");
	std::vector<double> &cv = bag.reals("trst_cov");
	off.clear(); ex.clear(); me.clear(); cv.clear();
	off.push_back(0);
	for(size_t i = 0; i < v.size(); i++)
	{
		for(size_t k = 0; k < v[i].exons.size(); k++) { ex.push_back(v[i].exons[k].first); ex.push_back(v[i].exons[k].second); }
		off.push_back((int32_t)ex.size() / 2);
		me.push_back((int32_t)v[i].strand);
		cv.push_back(v[i].coverage);
	}
}

// the lines of assembler::assemble(bundle&) between transform and assemble(gr, ps, sid) (meta/assembler.cc:113-141)
void seed_edge_support(splice_graph &gr, int sample_id)
{
	PEEI pei = gr.edges();
	for(edge_iterator it = pei.first; it != pei.second; it++)
	{
		edge_descriptor e = (*it);
		edge_info &ei = gr.get_editable_edge_info(e);
		ei.samples.insert(sample_id);
		ei.spAbd.insert(std::make_pair(sample_id, gr.get_edge_weight(e)));
		ei.abd = gr.get_edge_weight(e);
		ei.count = 1;
	}
}

} // namespace

// the reference end to end for one bundle that went through build_fragments + bridge (assembler::resolve, meta/assembler.cc:33-49):
// assembler::assemble(bundle&) = transform(bd, gr, true), build_phase_set, scallop.  Clears the bundle.
int ref_bundle_assemble(void *b, void *bagp)
{
	ref_handle *h = (ref_handle*)b;
	orc_bag &bag = *(orc_bag*)bagp;
	transcript_set tm(h->bd.chrm, 0, h->cfg.min_single_exon_clustering_overlap);
	std::mutex lock;
	assembler as(h->cfg, tm, lock, 0, 0, 0);
	as.assemble(h->bd);
	dump_transcripts(tm, bag);
	return (int)bag.reals("trst_cov").size();
}

// integration/adapter.cc, second half: bundle_base (mmap, splices, hcst, frgs, fcst), vector<pereads_cluster> and
// vector<bridge_path> rebuilt from the C-ABI views of bundle b, compared field by field with what the reference's own
// build_fragments + bundle::bridge steps leave (meta/bundle.cc:55-88) on a fresh handle of the same bundle.  Returns the number
// of differing fields (messages on stderr).
int ref_adapter_compare_bundle(void *hb, const agpu_evidence_view *ev, const agpu_fragments_view *fr, const agpu_cluster_view *cv,
		const agpu_bridge_view *bv, int b, int64_t hit_off)
{
	ref_handle *h = (ref_handle*)hb;
	bundle &bd = h->bd;
	bd.build_fragments();
	// bundle::bridge with its locals kept
	splice_graph gr;
	graph_builder gb(bd, h->cfg, h->sp);
	gb.build(gr);
	gr.build_vertex_index();
	std::vector<pereads_cluster> vc;
	graph_cluster gc(gr, bd, h->cfg.max_reads_partition_gap, false);
	gc.build_pereads_clusters(vc);
	bridge_solver bs(gr, vc, h->cfg, h->sp.insertsize_low, h->sp.insertsize_high);
	for(size_t k = 0; k < vc.size(); k++)
	{
		if(bs.opt[k].type <= 0) continue;
		bd.update_bridges(vc[k].frlist, bs.opt[k].chain, bs.opt[k].strand);
	}
	int bad = 0;
#define DIFF(cond, ...) do { if(cond) { if(bad < 5) { fprintf(stderr, "adapter_compare_bundle %d: ", b); fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); } bad++; } } while(0)
	auto far = [](double x, double y) { return fabs(x - y) > 1e-9 * std::max(fabs(x), 1e-300) && x != y; };
	// ---- bundle_base
	bundle_base bb;
	bb.hits = bd.hits;
	std::vector<uint8_t> xs(bd.hits.size());
	for(size_t i = 0; i < bd.hits.size(); i++) xs[i] = (uint8_t)bd.hits[i].xs;
	DIFF(agpu_adapter_bundle(ev, fr, b, hit_off, xs.data(), bb) != 0, "adapter_bundle failed");
	DIFF(bb.lpos != bd.lpos || bb.rpos != bd.rpos || bb.strand != bd.strand, "bounds / strand");
	DIFF(bb.splices != bd.splices, "splices");
	{
		SIMI i1 = bd.mmap.begin(), i2 = bb.mmap.begin();
		int n = 0;
		for(; i1 != bd.mmap.end() && i2 != bb.mmap.end(); ++i1, ++i2, ++n)
			DIFF(lower(i1->first) != lower(i2->first) || upper(i1->first) != upper(i2->first) || i1->second != i2->second, "mmap segment %d", n);
		DIFF(i1 != bd.mmap.end() || i2 != bb.mmap.end(), "mmap length");
	}
	auto same_chain_set = [&](const chain_set &a, const chain_set &c, const char *what, bool handles_xs)
	{
		DIFF(a.chains.size() != c.chains.size(), "%s groups %d vs %d", what, (int)a.chains.size(), (int)c.chains.size());
		for(size_t i = 0; i < a.chains.size() && i < c.chains.size(); i++)
		{
			DIFF(a.chains[i].size() != c.chains[i].size(), "%s group %d size", what, (int)i);
			for(size_t j = 0; j < a.chains[i].size() && j < c.chains[i].size(); j++)
				DIFF(a.chains[i][j].first != c.chains[i][j].first || a.chains[i][j].second != c.chains[i][j].second, "%s chain %d.%d", what, (int)i, (int)j);
		}
		DIFF(a.pmap != c.pmap, "%s pmap", what);
		DIFF(a.hmap.size() != c.hmap.size(), "%s hmap size %d vs %d", what, (int)a.hmap.size(), (int)c.hmap.size());
		for(std::map<int, AI3>::const_iterator it = a.hmap.begin(); it != a.hmap.end(); ++it)
		{
			std::map<int, AI3>::const_iterator jt = c.hmap.find(it->first);
			DIFF(jt == c.hmap.end(), "%s handle %d missing", what, it->first);
			if(jt == c.hmap.end()) continue;
			DIFF(it->second[0] != jt->second[0] || it->second[1] != jt->second[1], "%s handle %d -> %d.%d vs %d.%d", what, it->first,
					it->second[0], it->second[1], jt->second[0], jt->second[1]);
			if(handles_xs) DIFF(it->second[2] != jt->second[2], "%s handle %d xs class", what, it->first);
		}
	};
	same_chain_set(bd.hcst, bb.hcst, "hcst", true);
	same_chain_set(bd.fcst, bb.fcst, "fcst", false);
	DIFF(bb.frgs != bd.frgs, "frgs");
	// ---- vector<pereads_cluster>: note the reference's clusters were built BEFORE update_bridges changed frgs; so were the device's
	std::vector<pereads_cluster> vc2;
	agpu_adapter_clusters(cv, &ev->hcst, b, vc2);
	DIFF(vc.size() != vc2.size(), "clusters %d vs %d", (int)vc.size(), (int)vc2.size());
	for(size_t k = 0; k < vc.size() && k < vc2.size(); k++)
	{
		DIFF(vc[k].chain1 != vc2[k].chain1 || vc[k].chain2 != vc2[k].chain2, "cluster %d chains", (int)k);
		DIFF(vc[k].bounds != vc2[k].bounds || vc[k].extend != vc2[k].extend, "cluster %d bounds / extend", (int)k);
		DIFF(vc[k].frlist != vc2[k].frlist || vc[k].count != vc2[k].count, "cluster %d frlist / count", (int)k);
	}
	// ---- vector<bridge_path>
	std::vector<bridge_path> opt2;
	agpu_adapter_bridges(bv, cv, b, opt2);
	DIFF(bs.opt.size() != opt2.size(), "bridge paths %d vs %d", (int)bs.opt.size(), (int)opt2.size());
	for(size_t k = 0; k < bs.opt.size() && k < opt2.size(); k++)
	{
		const bridge_path &a = bs.opt[k], &c = opt2[k];
		DIFF(a.type != c.type, "opt %d type %d vs %d", (int)k, a.type, c.type);
		DIFF(a.strand != c.strand || a.choices != c.choices, "opt %d strand / choices", (int)k);
		DIFF(far(a.score, c.score), "opt %d score %f vs %f", (int)k, a.score, c.score);
		DIFF(a.chain != c.chain || a.whole != c.whole, "opt %d chain / whole", (int)k);
	}
#undef DIFF
	return bad;
}



// everything scallop reads: the reference's own transform(bd, gr, true) + build_phase_set on the handle's bundle against the
// graph and phase set the adapter rebuilds from the views, field by field.  Returns the number of differences (first few on
// stderr); the stub vertices' maxcov, which the reference leaves uninitialised, is not compared.
int ref_adapter_compare(void *hb, const agpu_graph_view *g, const agpu_revise_view *r, const agpu_phase_view *p, int b)
{
	ref_handle *h = (ref_handle*)hb;
	transcript_set tm(h->bd.chrm, 0, h->cfg.min_single_exon_clustering_overlap);
	std::mutex lock;
	assembler as(h->cfg, tm, lock, 0, 0, 0);
	h->bd.set_gid(0, 0, 0, 0);
	splice_graph g1, g2;
	as.transform(h->bd, g1, true);
	phase_set p1, p2;
	h->bd.build_phase_set(p1, g1);
	if(agpu_adapter_graph(g, r, b, h->bd.chrm, h->bd.gid, g2) != 0) return -1;
	agpu_adapter_phase_set(p, b, p2);
	int bad = 0;
#define DIFF(cond, ...) do { if(cond) { if(bad < 5) { fprintf(stderr, "adapter_compare bundle %d: ", b); fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); } bad++; } } while(0)
	auto far = [](double x, double y) { return fabs(x - y) > 1e-9 * std::max(fabs(x), 1e-300) && x != y; };
	DIFF(g1.strand != g2.strand, "strand %c vs %c", g1.strand, g2.strand);
	DIFF(g1.chrm != g2.chrm || g1.gid != g2.gid, "chrm / gid");
	DIFF(g1.num_vertices() != g2.num_vertices(), "vertices %d vs %d", (int)g1.num_vertices(), (int)g2.num_vertices());
	DIFF(g1.num_edges() != g2.num_edges(), "edges %d vs %d", (int)g1.num_edges(), (int)g2.num_edges());
	if(bad) return bad;
	const int v0 = g->vert_off[b];
	for(int x = 0; x < (int)g1.num_vertices(); x++)
	{
		const vertex_info &a = g1.get_vertex_info(x), &c = g2.get_vertex_info(x);
		DIFF(far(g1.get_vertex_weight(x), g2.get_vertex_weight(x)), "vertex %d weight", x);
		DIFF(a.lpos != c.lpos || a.rpos != c.rpos || a.length != c.length || a.type != c.type || a.regional != c.regional, "vertex %d ints", x);
		DIFF(a.pos != c.pos || a.sdist != c.sdist || a.tdist != c.tdist || a.count != c.count || a.lstrand != c.lstrand || a.rstrand != c.rstrand,
				"vertex %d defaults", x);
		DIFF(far(a.stddev, c.stddev), "vertex %d stddev", x);
		if(g->vert_d[3 * (size_t)(v0 + x) + 2] >= 0) DIFF(far(a.maxcov, c.maxcov), "vertex %d maxcov %f vs %f", x, a.maxcov, c.maxcov);
		DIFF(a.unbridge_leaving_count != c.unbridge_leaving_count || a.unbridge_coming_count != c.unbridge_coming_count, "vertex %d unbridge counts", x);
		DIFF(far(a.unbridge_leaving_ratio, c.unbridge_leaving_ratio) || far(a.unbridge_coming_ratio, c.unbridge_coming_ratio), "vertex %d unbridge ratios", x);
		DIFF(far(a.boundary_loss1, c.boundary_loss1) || far(a.boundary_loss2, c.boundary_loss2) || far(a.boundary_loss3, c.boundary_loss3)
				|| far(a.boundary_merged_loss, c.boundary_merged_loss), "vertex %d boundary_loss", x);
		DIFF(g1.in_degree(x) != g2.in_degree(x) || g1.out_degree(x) != g2.out_degree(x), "vertex %d degrees", x);
	}
	// splice_graph::edges() is ordered by edge address; the out-edge sets are ordered by (source, target)
	for(int x = 0; x < (int)g1.num_vertices(); x++)
	{
	PEEI e1 = g1.out_edges(x), e2 = g2.out_edges(x);
	edge_iterator i1 = e1.first, i2 = e2.first;
	for(; i1 != e1.second && i2 != e2.second; ++i1, ++i2)
	{
		const edge_info &a = g1.get_edge_info(*i1), &c = g2.get_edge_info(*i2);
		DIFF((*i1)->source() != (*i2)->source() || (*i1)->target() != (*i2)->target(), "edge %d->%d vs %d->%d", (*i1)->source(), (*i1)->target(),
				(*i2)->source(), (*i2)->target());
		DIFF(far(g1.get_edge_weight(*i1), g2.get_edge_weight(*i2)), "edge %d->%d weight", (*i1)->source(), (*i1)->target());
		DIFF(far(a.weight, c.weight) || a.strand != c.strand, "edge %d->%d info weight %f vs %f strand %d vs %d", (*i1)->source(), (*i1)->target(),
				a.weight, c.weight, a.strand, c.strand);
		DIFF(a.length != c.length || a.type != c.type || a.jid != c.jid || a.count != c.count || far(a.stddev, c.stddev) || far(a.abd, c.abd)
				|| far(a.confidence, c.confidence), "edge %d->%d info defaults", (*i1)->source(), (*i1)->target());
	}
	}
	DIFF(p1.pmap != p2.pmap, "phase set: %d vs %d lists", (int)p1.pmap.size(), (int)p2.pmap.size());
#undef DIFF
	return bad;
}

// the same with the graph and the phase set rebuilt from the C-ABI views by integration/adapter.cc: what the reference's
// assembler does once transform / build_phase_set are replaced by the adapter calls
int ref_adapter_assemble(const agpu_graph_view *g, const agpu_revise_view *r, const agpu_phase_view *p, int b, int n_frgs, int sample_id,
		const orc_params *prm, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	parameters cfg;
	sample_profile sp(sample_id, 1000000);
	apply_params(prm, cfg, sp);
	transcript_set tm("chr", 0, cfg.min_single_exon_clustering_overlap);
	std::mutex lock;
	assembler as(cfg, tm, lock, 0, 0, 0);
	splice_graph gr;
	if(agpu_adapter_graph(g, r, b, "chr", "instance.0.0.0.0", gr) != 0) return -1;
	gr.reads = n_frgs;
	gr.subgraph = 1;
	seed_edge_support(gr, sample_id);
	phase_set ps;
	agpu_adapter_phase_set(p, b, ps);
	as.assemble(gr, ps, sample_id);
	dump_transcripts(tm, bag);
	return (int)bag.reals("trst_cov").size();
}

// previewer::infer_library_type (meta/previewer.cc:29-148) over the records served by the htslib stand-in; dumps "preview" =
// library_type, bam_with_xs, num_xs, spn
int ref_infer_library_type(const orc_records_in *in, const orc_params *prm, int max_preview_reads, int max_preview_spliced_reads,
		int min_preview_spliced_reads, double preview_infer_ratio, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	parameters cfg;
	sample_profile sp(0, 1000000);
	apply_params(prm, cfg, sp);
	cfg.max_preview_reads = max_preview_reads; cfg.max_preview_spliced_reads = max_preview_spliced_reads;
	cfg.min_preview_spliced_reads = min_preview_spliced_reads; cfg.preview_infer_ratio = preview_infer_ratio;
	hts_shim_file file;
	for(int k = 0; k < in->n_chrom; k++)
	{
		file.target_name.push_back("chr" + std::to_string(k + 1));
		file.target_len.push_back((uint32_t)in->chrom_len[k]);
	}
	for(int64_t i = 0; i < in->n; i++)
	{
		uint32_t c0 = in->cigar_off[i], c1 = in->cigar_off[i + 1];
		file.records.push_back(hts_shim_make_record(in->tid[i], in->pos[i], in->mapq[i], in->flag[i], in->tid[i], in->mpos[i], in->isize[i],
				qname_of(in->qid[i]), in->cigar + c0, c1 - c0, (char)in->xs[i], '.', 1, 1, -1));
	}
	char name[64];
	snprintf(name, sizeof(name), "mem:prev:%p", (const void*)in);
	hts_shim_register(name, file);
	sp.align_file = name;
	previewer pv(cfg, sp);
	pv.infer_library_type();
	std::vector<int32_t> &o = bag.ints("preview");
	o.clear();
	o.push_back(sp.library_type); o.push_back(sp.bam_with_xs); o.push_back(sp.num_xs); o.push_back(sp.spn);
	hts_shim_clear();
	return sp.library_type;
}

// previewer::infer_insertsize (meta/previewer.cc:151-304) over the same records through the htslib stand-in: the reference's own
// record loop, bundle_base (with its never-flushed interval buffer), build_fragments, graph_builder, graph_cluster and histogram.
// "isize" = insert_total, insertsize_low, insertsize_high, insertsize_median; "isize_d" = insertsize_ave, insertsize_std
int ref_infer_insertsize(const orc_records_in *in, const orc_params *prm, int max_preview_reads, int min_preview_spliced_reads,
		int min_num_hits_in_bundle, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	parameters cfg;
	sample_profile sp(0, 1000000);
	apply_params(prm, cfg, sp);
	cfg.max_preview_reads = max_preview_reads; cfg.min_preview_spliced_reads = min_preview_spliced_reads;
	cfg.min_num_hits_in_bundle = min_num_hits_in_bundle;
	hts_shim_file file;
	for(int k = 0; k < in->n_chrom; k++)
	{
		file.target_name.push_back("chr" + std::to_string(k + 1));
		file.target_len.push_back((uint32_t)in->chrom_len[k]);
	}
	for(int64_t i = 0; i < in->n; i++)
	{
		uint32_t c0 = in->cigar_off[i], c1 = in->cigar_off[i + 1];
		file.records.push_back(hts_shim_make_record(in->tid[i], in->pos[i], in->mapq[i], in->flag[i], in->tid[i], in->mpos[i], in->isize[i],
				qname_of(in->qid[i]), in->cigar + c0, c1 - c0, (char)in->xs[i], '.', 1, 1, -1));
	}
	char name[64];
	snprintf(name, sizeof(name), "mem:isz:%p", (const void*)in);
	hts_shim_register(name, file);
	sp.align_file = name;
	sp.insert_total = 0;
	previewer pv(cfg, sp);
	pv.infer_insertsize();
	std::vector<int32_t> &o = bag.ints("isize");
	o.clear();
	o.push_back(sp.insert_total); o.push_back(sp.insertsize_low); o.push_back(sp.insertsize_high); o.push_back(sp.insertsize_median);
	std::vector<double> &d = bag.reals("isize_d");
	d.clear();
	d.push_back(sp.insertsize_ave); d.push_back(sp.insertsize_std);
	hts_shim_clear();
	return sp.insert_total;
}


// generator::resolve + generator::generate (meta/generator.cc:51-227) on an in-memory file behind the htslib stand-in: one
// region per chromosome that starts at its first record (start_off is a record index in the stand-in's bgzf_seek)
int ref_generate(const orc_records_in *in, const orc_params *prm, int use_second_alignment, void *bagp)
{
	return ref_generate_regions(in, prm, use_second_alignment, 0, bagp);
}

// region_length > 0: the table comes from the reference's own sample_profile::set_batch_boundaries (dumped as reg_off /
// reg_start1 / reg_start2 / reg_end1 / reg_start_off) and one generator::resolve runs per region with start1 < end1, like
// incubator::generate (meta/incubator.cc:355-380)
int ref_generate_regions(const orc_records_in *in, const orc_params *prm, int use_second_alignment, int region_length, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	parameters cfg;
	sample_profile sp(0, region_length > 0 ? region_length : 1000000);
	apply_params(prm, cfg, sp);
	cfg.use_second_alignment = use_second_alignment != 0;
	hts_shim_file file;
	for(int k = 0; k < in->n_chrom; k++)
	{
		file.target_name.push_back("chr" + std::to_string(k + 1));
		file.target_len.push_back((uint32_t)in->chrom_len[k]);
	}
	std::vector<int64_t> first(in->n_chrom, -1);
	for(int64_t i = 0; i < in->n; i++)
	{
		uint32_t c0 = in->cigar_off[i], c1 = in->cigar_off[i + 1];
		file.records.push_back(hts_shim_make_record(in->tid[i], in->pos[i], in->mapq[i], in->flag[i], in->tid[i], in->mpos[i], in->isize[i],
				qname_of(in->qid[i]), in->cigar + c0, c1 - c0, (char)in->xs[i], '.', 1, 1, -1));
		if(in->tid[i] >= 0 && in->tid[i] < in->n_chrom && first[in->tid[i]] < 0) first[in->tid[i]] = i;
	}
	char name[64];
	snprintf(name, sizeof(name), "mem:%p", (const void*)in);
	hts_shim_register(name, file);
	sp.align_file = name;
	sp.start1.assign(in->n_chrom, std::vector<int32_t>(1, 0));
	sp.start2.assign(in->n_chrom, std::vector<int32_t>(1, 0));
	sp.end1.assign(in->n_chrom, std::vector<int32_t>(1, 0x7fffffff));
	sp.end2.assign(in->n_chrom, std::vector<int32_t>(1, 0x7fffffff));
	sp.start_off.assign(in->n_chrom, std::vector<off_t>(1, 0));
	std::vector<int32_t> &off = bag.ints("gen_off"), &gb = bag.ints("gen_bundle");
	std::vector<int32_t> &gp = bag.ints("gen_pos"), &gr = bag.ints("gen_rpos"), &gm = bag.ints("gen_mpos"), &gi = bag.ints("gen_isize");
	std::vector<int32_t> &gf = bag.ints("gen_flag"), &gs = bag.ints("gen_strand"), &gx = bag.ints("gen_xs");
	off.clear(); gb.clear(); gp.clear(); gr.clear(); gm.clear(); gi.clear(); gf.clear(); gs.clear(); gx.clear();
	off.push_back(0);
	int nb = 0;
	if(region_length > 0)
	{
		sp.set_batch_boundaries(cfg.min_bundle_gap, cfg.max_read_span);
		std::vector<int32_t> &ro = bag.ints("reg_off"), &r1 = bag.ints("reg_start1"), &r2 = bag.ints("reg_start2"), &re = bag.ints("reg_end1");
		std::vector<int32_t> &rs = bag.ints("reg_start_off");
		ro.clear(); r1.clear(); r2.clear(); re.clear(); rs.clear();
		ro.push_back(0);
		for(size_t t = 0; t < sp.start1.size(); t++)
		{
			for(size_t k = 0; k < sp.start1[t].size(); k++)
			{
				r1.push_back(sp.start1[t][k]); r2.push_back(sp.start2[t][k]); re.push_back(sp.end1[t][k]); rs.push_back((int32_t)sp.start_off[t][k]);
			}
			ro.push_back((int32_t)r1.size());
		}
	}
	for(int t = 0; t < in->n_chrom; t++)
	for(size_t rid = 0; rid < sp.start1[t].size(); rid++)
	{
		if(region_length <= 0)
		{
			if(first[t] < 0) continue;
			sp.start_off[t][0] = (off_t)first[t];
		}
		else if(sp.start1[t][rid] >= sp.end1[t][rid]) continue;
		std::vector<bundle> vcb;
		{
			generator gt(sp, vcb, cfg, t, (int)rid);
			gt.resolve();
		}
		for(size_t k = 0; k < vcb.size(); k++)
		{
			bundle &bd = vcb[k];
			gb.push_back(bd.tid); gb.push_back(bd.lpos); gb.push_back(bd.rpos); gb.push_back((int32_t)bd.strand);
			for(size_t i = 0; i < bd.hits.size(); i++)
			{
				const hit &h = bd.hits[i];
				gp.push_back(h.pos); gr.push_back(h.rpos); gm.push_back(h.mpos); gi.push_back(h.isize); gf.push_back(h.flag);
				gs.push_back((int32_t)h.strand); gx.push_back((int32_t)h.xs);
			}
			off.push_back((int32_t)gp.size());
			nb++;
		}
	}
	hts_shim_clear();
	return nb;
}

int ref_group_bridge(void **bs, int n, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	if(n < 2) return -1;
	ref_handle *h0 = (ref_handle*)bs[0];
	// meta/assembler.cc:977-987
	bundle cb(h0->cfg, h0->sp);
	cb.copy_meta_information(h0->bd);
	// meta/assembler.cc:152-175 (combine_bundles)
	std::vector<PI> v;
	for(int k = 0; k < n; k++)
	{
		bundle &g = ((ref_handle*)bs[k])->bd;
		v.push_back(PI(k, std::distance(g.mmap.begin(), g.mmap.end())));
	}
	sort(v.begin(), v.end(), [](const PI &x, const PI &y){ return x.second > y.second; });
	std::vector<int32_t> &ord = bag.ints("combine_order");
	ord.clear();
	for(size_t i = 0; i < v.size(); i++)
	{
		cb.combine(((ref_handle*)bs[v[i].first])->bd, true);
		ord.push_back(v[i].first);
	}
	dump_chain_set(cb.hcst, bag, "cb_hcst", 0, "cb_hit_chain");
	dump_chain_set(cb.fcst, bag, "cb_fcst", 0, "cb_frg_chain");
	dump_segments(cb.mmap, bag, "cb_seg");
	std::vector<int32_t> &cbb = bag.ints("cb_bundle");
	cbb.clear();
	cbb.push_back(cb.lpos); cbb.push_back(cb.rpos); cbb.push_back((int32_t)cb.strand);

	splice_graph gr;
	graph_builder gb(cb, h0->cfg, cb.sp);
	gb.build(gr);
	gr.build_vertex_index();
	dump_graph(gr, h0->cfg, bag, "cb_", dump_builder(gb, h0->cfg, bag, "cb_"));

	int total = 0;
	for(int k = 0; k < n; k++)
	{
		ref_handle *h = (ref_handle*)bs[k];
		char pre[32];
		snprintf(pre, sizeof(pre), "b%d_", k);
		total += cluster_solve_update(gr, h->bd, h0->cfg, bag, pre, true);
	}
	return total;
}

int ref_bundle_set_sample(void *b, int sample_id)
{
	((ref_handle*)b)->sp.sample_id = sample_id;
	return 0;
}

namespace {

// per-edge support and per-vertex boundary losses of one graph, edges in out-edge order:
// <pre>sup_edge = src dst count per edge, <pre>sup_abd = abd per edge, <pre>sup_off / <pre>sup_sample / <pre>sup_sabd = the
// (sample, abundance) entries of spAbd per edge sorted by sample, <pre>sup_set_off / <pre>sup_set = ei.samples per edge,
// <pre>sup_loss = boundary_loss1 boundary_loss2 boundary_loss3 boundary_merged_loss per vertex
void dump_support(splice_graph &gr, orc_bag &bag, const std::string &pre)
{
	std::vector<int32_t> &se = bag.ints(pre + "sup_edge"), &so = bag.ints(pre + "sup_off"), &ss = bag.ints(pre + "sup_sample");
	std::vector<int32_t> &to = bag.ints(pre + "sup_set_off"), &ts = bag.ints(pre + "sup_set");
	std::vector<double> &sa = bag.reals(pre + "sup_abd"), &sb = bag.reals(pre + "sup_sabd"), &sl = bag.reals(pre + "sup_loss");
	se.clear(); so.clear(); ss.clear(); to.clear(); ts.clear(); sa.clear(); sb.clear(); sl.clear();
	so.push_back(0); to.push_back(0);
	for(int i = 0; i < (int)gr.num_vertices(); i++)
	{
		const vertex_info &vi = gr.get_vertex_info(i);
		sl.push_back(vi.boundary_loss1); sl.push_back(vi.boundary_loss2); sl.push_back(vi.boundary_loss3); sl.push_back(vi.boundary_merged_loss);
		PEEI pe = gr.out_edges(i);
		for(edge_iterator it = pe.first; it != pe.second; ++it)
		{
			const edge_info &ei = gr.get_edge_info(*it);
			se.push_back((*it)->source()); se.push_back((*it)->target()); se.push_back(ei.count);
			sa.push_back(ei.abd);
			std::map<int, double> m(ei.spAbd.begin(), ei.spAbd.end());
			for(std::map<int, double>::iterator z = m.begin(); z != m.end(); ++z) { ss.push_back(z->first); sb.push_back(z->second); }
			so.push_back((int32_t)ss.size());
			ts.insert(ts.end(), ei.samples.begin(), ei.samples.end());
			to.push_back((int32_t)ts.size());
		}
	}
}

} // namespace

// the cross-sample support features of assembler::assemble(vector<bundle*>) (meta/assembler.cc:177-373) on bundles that went
// through build_fragments, bundle::bridge and assembler::bridge: the loops of that function restated around the reference's own
// transform / junction_support / start_end_support / non_splicing_support / boundary_extend / fix_missing_edges / assemble.
// Member k is dumped ("m<k>_" prefix) at the point where the reference assembles it, the combined graph ("x_") at the end.
// ORC_SUPPORT_NO_ASSEMBLE=1 leaves the assemble(gr, ps, sid) calls out (to show what they change for the later members).
int ref_group_support(void **bs, int n, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	if(n < 2) return -1;
	ref_handle *h0 = (ref_handle*)bs[0];
	std::vector<bundle*> gv;
	for(int k = 0; k < n; k++) gv.push_back(&((ref_handle*)bs[k])->bd);
	transcript_set tm(h0->bd.chrm, 0, h0->cfg.min_single_exon_clustering_overlap);
	std::mutex lock;
	assembler as(h0->cfg, tm, lock, 0, 0, 0);
	int subindex = 0;
	bundle bx(h0->cfg, gv[0]->sp);
	bx.copy_meta_information(*(gv[0]));
	as.combine_bundles(bx, gv);
	bx.set_gid(0, 0, 0, subindex++);
	splice_graph gx;
	as.transform(bx, gx, false);
	gx.reads = bx.frgs.size();
	gx.subgraph = gv.size();
	std::unordered_map<int64_t, std::set<int> > junc2sup;
	std::unordered_map<int64_t, std::unordered_map<int, double> > sup2abd;
	phase_set px;
	{
		PEEI pei = gx.edges();
		for(edge_iterator it = pei.first; it != pei.second; it++)
		{
			edge_descriptor e = *it;
			int s = e->source(), t = e->target();
			edge_info &ei = gx.get_editable_edge_info(e);
			ei.samples.clear(); ei.spAbd.clear();
			ei.samples.insert(-1);
			ei.spAbd.insert(std::make_pair(-1, gx.get_edge_weight(e)));
			ei.abd = gx.get_edge_weight(e);
			ei.count = 1;
			if(s == 0 || t == (int)gx.num_vertices() - 1) continue;
			if(gx.get_vertex_info(s).rpos == gx.get_vertex_info(t).lpos) continue;
			int64_t p = pack(gx.get_vertex_info(s).rpos, gx.get_vertex_info(t).lpos);
			junc2sup[p].insert(-1);
			sup2abd[p].insert(std::make_pair(-1, gx.get_edge_weight(e)));
		}
	}
	std::vector<splice_graph*> grv;
	for(int k = 0; k < n; k++)
	{
		bundle &bd = *(gv[k]);
		bd.set_gid(0, 0, 0, subindex++);
		splice_graph *grp = new splice_graph();
		grv.push_back(grp);
		splice_graph &gr = *grp;
		as.transform(bd, gr, true);
		gr.reads = bd.frgs.size();
		gr.subgraph = gv.size();
		PEEI pei = gr.edges();
		for(edge_iterator it = pei.first; it != pei.second; it++)
		{
			edge_descriptor e = *it;
			int s = e->source(), t = e->target();
			edge_info &ei = gr.get_editable_edge_info(e);
			ei.samples.clear(); ei.spAbd.clear();
			ei.samples.insert(bd.sp.sample_id);
			ei.spAbd.insert(std::make_pair(bd.sp.sample_id, gr.get_edge_weight(e)));
			ei.abd = gr.get_edge_weight(e);
			ei.count = 1;
			if(s == 0 || t == (int)gr.num_vertices() - 1) continue;
			if(gr.get_vertex_info(s).rpos == gr.get_vertex_info(t).lpos) continue;
			int64_t p = pack(gr.get_vertex_info(s).rpos, gr.get_vertex_info(t).lpos);
			junc2sup[p].insert(bd.sp.sample_id);
			sup2abd[p].insert(std::make_pair(bd.sp.sample_id, gr.get_edge_weight(e)));
		}
	}
	for(int k = 0; k < n; k++)
	{
		bundle &bd = *(gv[k]);
		splice_graph &gr = *(grv[k]);
		as.fix_missing_edges(gr, gx);
		as.junction_support(gr, junc2sup, sup2abd);
		for(int j = 0; j < n; j++)
		{
			bundle &bd1 = *(gv[j]);
			splice_graph &gr1 = *(grv[j]);
			as.start_end_support(bd1.sp.sample_id, gr1, gr);
			as.non_splicing_support(bd1.sp.sample_id, gr1, gr);
			as.boundary_extend(bd1.sp.sample_id, gr, gr1, 1);
			as.boundary_extend(bd1.sp.sample_id, gr, gr1, 2);
			as.boundary_extend(bd1.sp.sample_id, gr, gr1, 3);
		}
		as.start_end_support(bd.sp.sample_id, gr, gx);
		as.non_splicing_support(bd.sp.sample_id, gr, gx);
		as.boundary_extend(-1, gr, gx, 1);
		char pre[32];
		snprintf(pre, sizeof(pre), "m%d_", k);
		dump_support(gr, bag, pre);
		// the reference assembles the member here; assemble(gr, ps, sid) regroups the start / end boundaries of gr
		// (group_start_boundaries / group_end_boundaries, rnacore/graph_reviser.cc:916-1066) and extends its strands, so the
		// members after k see a MODIFIED graph of member k in their own rounds
		if(getenv("ORC_SUPPORT_GROUP_ONLY") != NULL)
		{
			// only the graph changes assemble(gr, ps, sid) makes BEFORE it hands gr to scallop (which then decomposes it in place)
			gr.extend_strands();
			std::map<int32_t, int32_t> smap, tmap;
			group_start_boundaries(gr, smap, h0->cfg.max_group_boundary_distance);
			group_end_boundaries(gr, tmap, h0->cfg.max_group_boundary_distance);
		}
		else if(getenv("ORC_SUPPORT_NO_ASSEMBLE") == NULL)
		{
			phase_set ps;
			bd.build_phase_set(ps, gr);
			px.combine(ps);
			as.assemble(gr, ps, bd.sp.sample_id);
		}
	}
	as.junction_support(gx, junc2sup, sup2abd);
	dump_support(gx, bag, "x_");
	for(int k = 0; k < n; k++) delete grv[k];
	return 0;
}

int ref_group_resolve(void **bs, int n, const orc_params *prm, void *bagp)
{
	orc_bag &bag = *(orc_bag*)bagp;
	parameters cfg;
	sample_profile sp(0, 1000000);
	apply_params(prm, cfg, sp);
	std::map<std::string, std::vector<PI> > sidx;
	bundle_group grp("chr", '.', 0, cfg, sidx);
	for(int k = 0; k < n; k++)
	{
		ref_handle *h = (ref_handle*)bs[k];
		bundle b(cfg, sp);
		b.chrm = "chr";
		b.strand = '.';
		b.tid = h->bd.tid;
		b.splices = h->bd.splices;
		grp.gset.push_back(b);
	}
	grp.resolve();
	std::vector<int32_t> &off = bag.ints("gvv_off");
	std::vector<int32_t> &val = bag.ints("gvv_val");
	off.clear(); val.clear();
	off.push_back(0);
	for(size_t i = 0; i < grp.gvv.size(); i++)
	{
		val.insert(val.end(), grp.gvv[i].begin(), grp.gvv[i].end());
		off.push_back((int32_t)val.size());
	}
	return 0;
}


// known-answer and randomised checks of the Boost.ICL stand-in (oracle/compat/boost/icl/interval_map.hpp), through the
// reference's own helpers (create_split, locate_boundary_iterators, compute_coverage, get_overlapped_length)
int ref_icl_kat(int32_t *out, int cap)
{
	int n = 0;
	// rnacore/interval_map.cc:320-331 (test_split_interval_map)
	split_interval_map imap;
	imap += make_pair(ROI(6, 7), 3);
	imap += make_pair(ROI(1, 3), 3);
	imap += make_pair(ROI(1, 2), 1);
	imap += make_pair(ROI(2, 5), 2);
	create_split(imap, 4);
	for(SIMI it = imap.begin(); it != imap.end() && n + 3 <= cap; it++) { out[n++] = lower(it->first); out[n++] = upper(it->first); out[n++] = it->second; }
	if(n < cap) out[n++] = -1;
	// coverage [i, j) for 0 <= i <= j <= 8 (:372-380)
	for(int i = 0; i <= 8; i++)
		for(int j = i; j <= 8; j++)
		{
			pair<SIMI, SIMI> p = locate_boundary_iterators(imap, i, j);
			if(n < cap) out[n++] = compute_coverage(imap, p.first, p.second);
		}
	if(n < cap) out[n++] = -1;
	// rnacore/interval_map.cc:435-451 (test_join_interval_map)
	join_interval_map m1, m2;
	m1 += make_pair(ROI(6, 7), 3);
	m1 += make_pair(ROI(1, 2), 1);
	m1 += make_pair(ROI(2, 5), 1);
	m2 += make_pair(ROI(1, 3), 3);
	m2 += make_pair(ROI(3, 4), 3);
	m2 += make_pair(ROI(5, 7), 1);
	if(n < cap) out[n++] = get_overlapped_length(m1, m2);
	if(n < cap) out[n++] = (int32_t)std::distance(m1.begin(), m1.end());
	if(n < cap) out[n++] = (int32_t)std::distance(m2.begin(), m2.end());
	if(n < cap) out[n++] = (int32_t)m1.size();          // ICL size() is the cardinality: 4 + 1
	return n;
}

// apply additions (l, r, v) to a split (join = 0) or joining (join = 1) map and dump its segments
int ref_icl_apply(int n, const int32_t *l, const int32_t *r, const int32_t *v, int join, int32_t *out, int cap)
{
	int k = 0;
	if(join)
	{
		join_interval_map m;
		for(int i = 0; i < n; i++) m += make_pair(ROI(l[i], r[i]), v[i]);
		for(JIMI it = m.begin(); it != m.end() && k + 3 <= cap; it++) { out[k++] = lower(it->first); out[k++] = upper(it->first); out[k++] = it->second; }
	}
	else
	{
		split_interval_map m;
		for(int i = 0; i < n; i++) m += make_pair(ROI(l[i], r[i]), v[i]);
		for(SIMI it = m.begin(); it != m.end() && k + 3 <= cap; it++) { out[k++] = lower(it->first); out[k++] = upper(it->first); out[k++] = it->second; }
	}
	return k;
}

// a script over two maps of the reference's types: op 0: A += (I, v); 1: A -= (I, v); 2: B += (I, v); 3: A += B (bundle::combine,
// meta/bundle.cc:102); 4: A -= every segment of B.  join selects join_interval_map, else split_interval_map.  Dumps A.
int ref_icl_script(int n, const int32_t *op, const int32_t *l, const int32_t *r, const int32_t *v, int join, int32_t *out, int cap)
{
	int k = 0;
	if(join)
	{
		join_interval_map A, B;
		for(int i = 0; i < n; i++)
		{
			if(op[i] == 0) A += make_pair(ROI(l[i], r[i]), v[i]);
			if(op[i] == 1) A -= make_pair(ROI(l[i], r[i]), v[i]);
			if(op[i] == 2) B += make_pair(ROI(l[i], r[i]), v[i]);
			if(op[i] == 3) A += B;
			if(op[i] == 4) for(JIMI it = B.begin(); it != B.end(); it++) A -= make_pair(it->first, it->second);
		}
		for(JIMI it = A.begin(); it != A.end() && k + 3 <= cap; it++) { out[k++] = lower(it->first); out[k++] = upper(it->first); out[k++] = it->second; }
	}
	else
	{
		split_interval_map A, B;
		for(int i = 0; i < n; i++)
		{
			if(op[i] == 0) A += make_pair(ROI(l[i], r[i]), v[i]);
			if(op[i] == 1) A -= make_pair(ROI(l[i], r[i]), v[i]);
			if(op[i] == 2) B += make_pair(ROI(l[i], r[i]), v[i]);
			if(op[i] == 3) A += B;
			if(op[i] == 4) for(SIMI it = B.begin(); it != B.end(); it++) A -= make_pair(it->first, it->second);
		}
		for(SIMI it = A.begin(); it != A.end() && k + 3 <= cap; it++) { out[k++] = lower(it->first); out[k++] = upper(it->first); out[k++] = it->second; }
	}
	return k;
}

}
