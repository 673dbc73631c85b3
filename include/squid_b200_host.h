/*
 * squid_b200 host twin — C entry points of the host-side stages that north_star keeps on the CPU:
 * decoding alignments into aligned blocks and loading the chimeric reads.
 *   sqh_open_case   = BuildRefName (src/ReadRec.cpp:267-283) + BuildChimericSBamRecord
 *                     (src/ReadRec.cpp:329-413) + the per-record ReadRec_t decode
 *                     (src/ReadRec.cpp:10-88) and tag / ChimName probes (src/SegmentGraph.cpp:297-302)
 *                     that the reference repeats inside each of its three BAM passes.
 * Inputs are BAM files (sqh_open_bam_case) or SQMB files (include/sqmb_format.h), the uncompressed BAM stand-in that
 * also feeds the test oracle's BamReader shim.
 */
#ifndef SQUID_B200_HOST_H
#define SQUID_B200_HOST_H
#include <stdint.h>
#include "squid_b200.h"
#ifdef __cplusplus
extern "C" {
#endif
typedef struct sqh_case sqh_case;
typedef struct sqh_options {   /* src/Config.cpp:18-28 */
    int32_t phred33;           /* Phred_Type: 1 => offset 33 (Config.cpp:19) */
    int32_t max_lowphred_len;  /* -pl */
    int32_t min_phred;         /* -pm */
    int32_t min_mapq;          /* -mq; < 0 => STAR default 255 (Config.cpp:221-222) */
    int32_t concord_dist_pos, concord_dist_idx;
} sqh_options;
void sqh_default_options(sqh_options *o);
int sqh_open_case(const char *concordant_sqmb, const char *chimeric_sqmb, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen);
/* The same from coordinate-sorted BAM files (BGZF-compressed or plain): replaces BamTools' BamReader::Open / GetHeader /
 * GetNextAlignment on the path (src/ReadRec.cpp:271-279, 340-343; src/SegmentGraph.cpp:293-296, 1570-1577, 3126-3129).
 * The file is inflated on all cores and decoded once for all three phases (SURVEY.md 8f row 1). */
int sqh_open_bam_case(const char *concordant_bam, const char *chimeric_bam, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen);
/* The chimeric BAM decoded as sqh_open_bam_case does, and only the header of the concordant BAM (ref_len, reference names): the
 * case's concordant batch is empty, because sqg_load_concordant_bam (squid_b200.h) decodes that file on the device.  config.read_len
 * and the chimeric reads come from the chimeric file. */
int sqh_open_bam_chimeric(const char *concordant_bam, const char *chimeric_bam, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen);
/* The ChimName list the concordant packer probes (the suffix-stripped Qnames of the chimeric reads plus the empty name,
 * src/SegmentGraph.cpp:196-201): *n names, name i = blob[off[i], off[i+1]).  Owned by the case. */
int sqh_case_chim_names(const sqh_case *c, const char **blob, const int64_t **off, int64_t *n);
/* The concordant file alone (SQMB), for a caller that already holds Chimrecord -- the binding of INTEGRATION.md
 * (integration/binding.cpp): chim_qnames[n_names] = the Qnames of Chimrecord, from which ChimName is built
 * (src/SegmentGraph.cpp:196-201).  The chimeric side of the case stays empty and config.read_len 0. */
int sqh_open_concordant(const char *concordant_sqmb, const char *const *chim_qnames, int64_t n_names, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen);
void sqh_close_case(sqh_case *c);
const sqg_batch *sqh_case_batch(const sqh_case *c);
sqg_chimeric *sqh_case_chimeric(sqh_case *c);
const sqg_config *sqh_case_config(const sqh_case *c);  /* read_len filled from the chimeric reads */
int32_t sqh_case_n_ref(const sqh_case *c);
const int32_t *sqh_case_ref_len(const sqh_case *c);
/* Known-answer access to the decoder: blocks of record r of the concordant table as
 * (ref_pos, match_ref, read_pos, match_read) rows; returns the block count. */
int32_t sqh_case_blocks(const sqh_case *c, int64_t r, int32_t *out4, int32_t max_blocks, int32_t *total_len, int32_t *lowphred_run);

/* Packs an sqg_batch into its wire form (squid_b200.h: sqg_wire) on all cores.  pinned != 0: the arrays are page-locked
 * (cudaHostAlloc) so that sqg_load_concordant_wire() copies them asynchronously.  SQG_EINVAL: aux >= 16, a record with more
 * than 65535 blocks or a decreasing blk_off.  Release with sqh_free_wire(). */
int sqh_pack_wire(const sqg_batch *batch, int32_t pinned, sqg_wire **out);
void sqh_free_wire(sqg_wire *w);
int64_t sqh_wire_bytes(const sqg_wire *w);

/*
 * Replaces SegmentGraph_t::ExactBreakpoint + CountTop (src/SegmentGraph.cpp:3019-3081, 51-102; SURVEY.md §8 row a17, host side).
 * The chimeric reads -- as sqg_build_edges left them, i.e. already trimmed once -- are located on the FINAL graph
 * (node_chr/pos/len[n_nodes]: the nodes after the host filters and compression, sorted, not necessarily tiling) with the
 * literal hinted scan of LocateRead (:1207-1293), which trims them in place again; every discordant split junction adds a
 * (bp1, bp2) pair to its edge and each edge keeps at most five representatives.
 * *rows6 = n_rows x (Ind1, Ind2, Head1, Head2, bp1, bp2) in the order of the reference's map<Edge_t, vector<pair>> (edges by
 * Edge_t::operator<, pairs in vector order); malloc'ed, release with sqh_free().
 */
int sqh_exact_breakpoint(const int32_t *node_chr, const int32_t *node_pos, const int32_t *node_len, int64_t n_nodes, sqg_chimeric *chim_inout,
                         int32_t concord_dist_pos, int32_t concord_dist_idx, int32_t **rows6, int64_t *n_rows);
void sqh_free(void *p);

/*
 * The two output formats of the path (SURVEY.md §8 row a20), byte for byte.
 *   sqh_write_graph  = SegmentGraph_t::OutputGraph (src/SegmentGraph.cpp:3223-3234): <prefix>_graph.txt
 *   sqh_write_bedpe  = DeMultiplyDisEdges (src/SegmentGraph.cpp:3012-3017) + WriteBEDPE (src/WriteIO.cpp:45-124): <prefix>_sv.txt.
 *                      Edges in vEdges order (weights still multiplied by -r); components = the ordering the ILP stage produced
 *                      (signed 1-based node ids, comp_off[n_comp + 1]); exactbp / support rows as sqh_exact_breakpoint returns
 *                      them / as ExactBPConcordantSupport fills its map (SegmentGraph.cpp:3171-3211).
 */
int sqh_write_graph(const char *path, const int32_t *chr, const int32_t *pos, const int32_t *len, const int32_t *support, const double *avg_depth,
                    const int32_t *label, int64_t n_nodes, const int32_t *ind1, const int32_t *ind2, const uint8_t *head1, const uint8_t *head2,
                    const int32_t *weight, int64_t n_edges);
int sqh_write_bedpe(const char *path, const char *const *ref_name, int32_t n_ref, const int32_t *chr, const int32_t *pos, const int32_t *len, int64_t n_nodes,
                    const int32_t *ind1, const int32_t *ind2, const uint8_t *head1, const uint8_t *head2, const int32_t *weight, int64_t n_edges,
                    const int64_t *comp_off, const int32_t *comp_nodes, int64_t n_comp, const int32_t *exactbp_rows6, int64_t n_exactbp,
                    const int32_t *support_rows6, int64_t n_support, double discordant_ratio, int32_t concord_dist_pos, int32_t concord_dist_idx);
#ifdef __cplusplus
}
#endif
#endif
