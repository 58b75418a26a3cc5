// TEST INFRASTRUCTURE ONLY (oracle/).  CPU restatement of the reference's per-bundle read-evidence
// path in plain sequential C++ over flat containers.  It restates the ALGORITHMS (each function cites the
// reference file:line it follows); it shares no code with aletsch_b200/ and none with /root/reference.
// Pinned against oracle/_ref (the reference's own translation units) by tests/test_oracle.py.
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this.
#ifndef ALETSCH_B200_ORACLE_RESTATE_H
#define ALETSCH_B200_ORACLE_RESTATE_H

#include <stdint.h>
#include <array>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "../orc_api.h"

namespace orc {

typedef std::array<int, 3> AI3;
typedef std::vector<int32_t> chain_t;

// rnacore/hit.h:66-97 (fields the path reads)
struct hit
{
	int32_t pos, rpos, mpos, isize;
	uint16_t flag;
	char strand, xs;
	uint64_t qid;
};

// rnacore/chain_set.h:18-35
struct chain_set
{
	std::map<int, AI3> hmap;                                      // handle -> (group, index, xs)
	std::map<int32_t, int> pmap;                                  // first coordinate -> group
	std::vector<std::vector<std::pair<chain_t, AI3> > > chains;   // insertion ordered
	void add(const chain_t &v, int h, char xs);
	void add(const chain_t &v, const AI3 &a);
	void add(const chain_set &cs);
	const chain_t *get(int h) const;
	std::vector<int32_t> get_splices() const;
};

// split_interval_map<int32, int32, partial_absorber> restricted to what the live path does with it:
// positive additions only.  Under positive-only additions every inserted interval end stays a segment
// border for ever and the value between two consecutive borders is the number of covering additions,
// so the map is fully described by a delta per position plus the set of borders.
struct coverage_map
{
	std::map<int32_t, int32_t> delta;      // position -> sum of (+v at starts, -v at ends); doubles as the border set
	void add(int32_t l, int32_t r, int32_t v);
	void add(const coverage_map &m);
	struct seg { int32_t l, r, c; };
	std::vector<seg> segments() const;     // [l, r) -> c > 0, in order
};

struct bundle
{
	int32_t tid, lpos, rpos;
	char strand;
	std::vector<hit> hits;
	std::vector<int> input_index;
	std::vector<AI3> frgs;
	std::vector<int32_t> splices;
	chain_set hcst, fcst;
	coverage_map mmap;
	orc_params prm;
	int sample = 0;                        // sample_profile::sample_id
};

struct junction { int32_t lpos, rpos; int count, xs0, xs1, xs2; char strand; int lexon, rexon; };
struct pexon { int32_t lpos, rpos; int ltype, rtype; double ave, dev, max, pvalue; bool stub; bool regional; };

struct edge { int s, t; double w; int strand; bool alive; };
struct graph
{
	char strand;
	std::vector<int32_t> vl, vr;
	std::vector<int> vlen, vtype, vregional;
	std::vector<double> vw, vdev, vmax;
	std::vector<edge> edges;                                 // insertion order
	std::vector<std::set<std::pair<int, int> > > out, in;    // (other endpoint, edge index), ordered like edge_base's (s, t) order
	std::map<int32_t, int> lindex, rindex;
	int nv() const { return (int)vl.size(); }
	int add_edge(int s, int t, double w, int strand);
	void remove_edge(int e);
	int find_edge(int s, int t) const;                       // edge index or -1
	void build_vertex_index();
	int locate_vertex(int32_t p) const;
};

struct cluster
{
	chain_t chain1, chain2;
	std::vector<int32_t> bounds, extend;
	std::vector<int> frlist;
	int count;
};

struct bridge_path
{
	int type, strand, choices;
	double score;
	std::vector<int> v, stack;
	chain_t chain, whole;
	bridge_path() : type(0), strand(0), choices(0), score(0) {}
};

struct revision
{
	std::vector<std::array<int, 2> > added;                  // boundary edges in the order they are added
	std::vector<double> added_w;
	std::vector<int> leave_cnt, come_cnt;                    // vertex_info::unbridge_* (rnacore/vertex_info.h:38-41)
	std::vector<double> leave_ratio, come_ratio;
};

// repeated_bounds: partial exons whose lpos or rpos an earlier one already has; link_partial_exons asserts there are none
// (rnacore/graph_builder.cc:255-258), so the graph is not the reference's when this is non-zero
struct builder_out { std::vector<junction> junctions; std::vector<pexon> pexons; int repeated_bounds = 0; };

void build_graph(const bundle &bd, graph &gr, builder_out &bo);
void build_phase_set(const bundle &bd, const graph &gr, std::map<chain_t, int> &ps);
void revise_graph(const bundle &bd, graph &gr, revision &rv);
void combine_bundles(bundle **bs, int n, bundle &cb, std::vector<int> *order);

// edge_info::samples / spAbd / abd / count and vertex_info::boundary_loss* of one graph (edges indexed like graph::edges)
struct support
{
	std::vector<std::set<int> > samples;
	std::vector<std::map<int, double> > spabd;
	std::vector<double> abd;
	std::vector<int> count;
	std::vector<std::array<double, 4> > loss;           // boundary_loss1, 2, 3, boundary_merged_loss per vertex
};
// one entry per member in grs / sups: the state at the point where the reference assembles that member
// returns -1 (and leaves the outputs partial) if a graph it builds has repeated partial-exon bounds
int group_support(bundle **bs, int n, std::vector<graph> &grs, std::vector<support> &sups, graph &gx, support &sx);
void build_fragments(bundle &bd);
void cluster_fragments(graph &gr, bundle &bd, std::vector<cluster> &vc);
void bridge_clusters(graph &gr, std::vector<cluster> &vc, const orc_params &prm, std::vector<bridge_path> &opt);
int update_bridges(bundle &bd, const std::vector<int> &frlist, const chain_t &chain, int strand);

} // namespace orc

#endif
