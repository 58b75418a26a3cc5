/* TEST INFRASTRUCTURE ONLY (oracle/).  Shared flat C interface of the two CPU checkers:
 *   - oracle/_ref/libaletsch_ref.so   the reference's own translation units, compiled
 *                                     unchanged from /root/reference (prefix "ref_")
 *   - oracle/liboracle.so             our CPU restatement of the same algorithms (prefix "orc_")
 * Both take the same packed bundle input and write results into a "bag" of named flat
 * arrays so that tests compare them array by array.  Nothing under aletsch_b200/ may
 * include, link or call this.
 */
#ifndef ALETSCH_B200_ORACLE_ORC_API_H
#define ALETSCH_B200_ORACLE_ORC_API_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* one bundle's hits, already routed to this strand bundle by the packer
 * (meta/generator.cc:87-179), in BAM order */
typedef struct orc_bundle_in
{
	int32_t n_hits;
	int32_t tid;
	const int32_t *pos;          /* [H] 0-based leftmost coordinate */
	const int32_t *mpos;         /* [H] mate position */
	const int32_t *isize;        /* [H] template length */
	const uint16_t *flag;        /* [H] BAM flag */
	const uint8_t *strand;       /* [H] hit.strand after set_strand + generator fix-up: '+','-','.' */
	const uint8_t *xs;           /* [H] hit.xs after set_tags: '+','-','.' */
	const uint64_t *qid;         /* [H] query-name key: equal keys <=> equal qnames */
	const uint32_t *cigar_off;   /* [H+1] offsets into cigar[] */
	const uint32_t *cigar;       /* raw BAM CIGAR ops, len<<4|op */
} orc_bundle_in;

/* decoded, coordinate-sorted records of one sample (what the BAM file holds), for the record loop of generator::resolve */
typedef struct orc_records_in
{
	int64_t n;
	int32_t n_chrom;
	const int32_t *chrom_len;
	const int32_t *tid, *pos, *mpos, *isize;
	const uint16_t *flag;
	const uint8_t *mapq;
	const uint8_t *xs;           /* goes into the record as an XS:A tag ('.': no tag) */
	const uint64_t *qid;
	const uint32_t *cigar_off;
	const uint32_t *cigar;
} orc_records_in;

/* the values of util/parameters.h + rnacore/sample_profile.h that the path reads */
typedef struct orc_params
{
	int32_t library_type;                 /* UNSTRANDED 0, FR_FIRST 1, FR_SECOND 2 */
	int32_t min_junction_support;
	int32_t normal_junction_threshold;
	int32_t extend_junction_threshold;
	int32_t min_subregion_gap;
	int32_t min_subregion_length;
	int32_t max_reads_partition_gap;
	int32_t bridge_end_relaxing;
	int32_t bridge_dp_solution_size;
	int32_t bridge_dp_stack_size;
	int32_t insertsize_low;
	int32_t insertsize_high;
	int32_t max_group_size;
	int32_t max_num_junctions_to_combine;
	double min_subregion_overlap;
	double min_guaranteed_edge_weight;
	double min_grouping_similarity;
	double max_grouping_similarity;
	double min_boundary_log_ratio;
	int32_t max_group_boundary_distance;  /* appended like agpu_params: the layouts stay equal */
} orc_params;

/* result bag: named flat arrays, kind 0 = int32, 1 = float64 */
void *orc_bag_new(void);
void orc_bag_free(void *bag);
void orc_bag_clear(void *bag);
int orc_bag_count(void *bag);
const char *orc_bag_name(void *bag, int i);
int orc_bag_kind(void *bag, int i);
int64_t orc_bag_len(void *bag, int i);
const void *orc_bag_data(void *bag, int i);

#define ORC_DECLARE(P) \
	void *P##_bundle_new(const orc_bundle_in *in, const orc_params *prm); \
	void P##_bundle_free(void *b); \
	int P##_bundle_evidence(void *b, void *bag); \
	int P##_bundle_fragments(void *b, void *bag); \
	int P##_bundle_graph(void *b, void *bag); \
	int P##_bundle_bridge(void *b, void *bag); \
	int P##_bundle_phase(void *b, void *bag); \
	int P##_bundle_revise(void *b, void *bag); \
	int P##_group_bridge(void **bs, int n, void *bag); \
	int P##_group_resolve(void **bs, int n, const orc_params *prm, void *bag);

/* restatement only: <P>_group_resolve on n given sorted splice lists (list k = list_val[list_off[k] .. list_off[k + 1])) instead of
 * bundle handles, so that constructed lists can be checked; "gvv_off" / "gvv_val" as there */
int orc_group_resolve_lists(int n, const int64_t *list_off, const int32_t *list_val, const orc_params *prm, void *bag);

/* reference build only: generator::resolve (meta/generator.cc:51-227) over the records served through the htslib stand-in;
 * dumps the bundles it creates (gen_off, gen_bundle = tid lpos rpos strand per bundle, gen_pos / rpos / mpos / isize / flag /
 * strand / xs per stored hit).  Returns the number of bundles. */
int ref_generate(const orc_records_in *in, const orc_params *prm, int use_second_alignment, void *bag);

/* reference build only: assembler::assemble(bundle&) end to end (transcripts: trst_off, trst_exon, trst_meta, trst_cov), and the
 * same with graph + phase set rebuilt from the C-ABI views through integration/adapter.cc (declared in ref_driver.cc; takes
 * agpu_graph_view / agpu_revise_view / agpu_phase_view pointers) */
int ref_bundle_assemble(void *b, void *bag);

/* reference build only: previewer::infer_library_type over the same records; "preview" = library_type, bam_with_xs, num_xs, spn */
int ref_infer_library_type(const orc_records_in *in, const orc_params *prm, int max_preview_reads, int max_preview_spliced_reads,
		int min_preview_spliced_reads, double preview_infer_ratio, void *bag);
/* reference build only: previewer::infer_insertsize over the same records; "isize" = insert_total, low, high, median; "isize_d" =
 * ave, std */
int ref_infer_insertsize(const orc_records_in *in, const orc_params *prm, int max_preview_reads, int min_preview_spliced_reads,
		int min_num_hits_in_bundle, void *bag);
/* Groundwork for SURVEY 8f-3 (nothing in the product implements this step yet).  <P>_bundle_set_sample: sample id of a bundle
 * handle (sample_profile::sample_id).  <P>_group_support: the cross-sample support features of assembler::assemble(vector<bundle*>)
 * (meta/assembler.cc:177-373) on bundles that went through fragments, bridge and group_bridge; member k is dumped at the point
 * where the reference assembles it (see dump_support in ref_driver.cc for the arrays).
 * ref_: the loops of that function around the reference's own member functions, INCLUDING assemble(gr, ps, sid) after every
 * member -- which hands the member's graph to scallop by reference, so the later members see it decomposed.  With
 * ORC_SUPPORT_GROUP_ONLY=1 only the graph changes assemble makes before scallop are applied (extend_strands,
 * group_start_boundaries, group_end_boundaries); with ORC_SUPPORT_NO_ASSEMBLE=1 none.
 * orc_: the restatement (restate/support.cc); it restates the GROUP_ONLY variant and is pinned against it. */
int ref_bundle_set_sample(void *b, int sample_id);
int ref_group_support(void **bs, int n, void *bag);
int orc_bundle_set_sample(void *b, int sample_id);
int orc_group_support(void **bs, int n, void *bag);
int ref_generate_regions(const orc_records_in *in, const orc_params *prm, int use_second_alignment, int region_length, void *bag);

/* reference build only -- timing entry for bench.py (cpu_baseline, --impl reference): records and hit objects are built by
 * ref_timing_new before any clock starts; ref_timing_run times add_hit_intervals + build_fragments + bundle::bridge() per bundle
 * on `threads` workers, no result dumps (see ref_driver.cc) */
void *ref_timing_new(int n_bundles, const orc_bundle_in *ins, const orc_params *prm);
void ref_timing_free(void *t);
int64_t ref_timing_hits(void *t);
int ref_timing_run(void *t, int threads, double *seconds, int64_t *bridged, int32_t *per_bundle_bridged);

ORC_DECLARE(ref)
ORC_DECLARE(orc)

#ifdef __cplusplus
}
#endif

#endif
