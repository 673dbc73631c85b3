/*
 * squid_b200 — C ABI of the B200-native segment-graph construction path of SQUID.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no FFI layer; its seam is four
 * member functions of SegmentGraph_t, called once per run from the constructor and main():
 *     BuildNode_STAR            src/SegmentGraph.h:77   (def. src/SegmentGraph.cpp:192)
 *     BuildEdges                src/SegmentGraph.h:79   (def. src/SegmentGraph.cpp:1932)
 *     ExactBPConcordantSupport  src/SegmentGraph.h:104  (def. src/SegmentGraph.cpp:3083)
 *     SegmentGraph_t(graphfile) src/SegmentGraph.h:71   (node reload, def. src/SegmentGraph.cpp:126)
 * Each entry point below names the reference interface it replaces.  INTEGRATION.md shows the
 * binding a SQUID maintainer adds to call them.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns 0 on success
 * or a negative SQG_E* code and never throws; a context is used by one host thread at a time;
 * input arrays are caller-owned HOST memory unless a function says DEVICE, and are not modified;
 * output arrays returned through `T**` are library-owned pinned host buffers that stay valid
 * until the next call of the same function on the same context or sqg_destroy().  There is no
 * CPU fallback: without a CUDA device sqg_create() fails with SQG_ENODEVICE.
 */
#ifndef SQUID_B200_H
#define SQUID_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SQG_OK 0
#define SQG_EINVAL (-1)     /* bad argument / malformed batch (unsorted, RefID out of range, ...) */
#define SQG_ENODEVICE (-2)  /* no usable CUDA device */
#define SQG_ECUDA (-3)      /* CUDA runtime error, see sqg_last_error() */
#define SQG_ESTATE (-4)     /* call order violated (e.g. build_edges before nodes exist) */
#define SQG_EUNSUPPORTED (-5) /* input the reference itself handles with undefined behaviour, or BWA mode */
#define SQG_ENOMEM (-6)

typedef struct sqg_ctx sqg_ctx;

/* The reference's Config globals that gate the path (src/Config.cpp:14-37). */
typedef struct sqg_config {
    int32_t using_star;        /* UsingSTAR        Config.cpp:18  (only 1 is implemented) */
    int32_t max_lowphred_len;  /* Max_LowPhred_Len Config.cpp:20  (-pl) */
    int32_t min_mapq;          /* Min_MapQual      Config.cpp:22, 221-222 (-mq; STAR default 255) */
    int32_t concord_dist_pos;  /* Concord_Dist_Pos Config.cpp:24  (-dp) */
    int32_t concord_dist_idx;  /* Concord_Dist_Idx Config.cpp:25  (-di) */
    int32_t read_len;          /* ReadLen          Config.cpp:14, set by BuildChimericSBamRecord ReadRec.cpp:378-379 */
} sqg_config;

/* aux bits of a record */
#define SQG_AUX_XA 1u        /* record.HasTag("XA")                       SegmentGraph.cpp:297 */
#define SQG_AUX_IH_GT1 2u    /* IH tag present with value > 1             SegmentGraph.cpp:298-302 */
#define SQG_AUX_CHIMNAME 8u  /* record.Name is in ChimName                SegmentGraph.cpp:302 */

/*
 * Struct-of-arrays batch of decoded alignment records, sorted by (ref_id, pos) (SURVEY.md App. B).
 * One record = one BAM alignment line.  Blocks are the gap-free aligned blocks that
 * ReadRec_t::ReadRec_t (src/ReadRec.cpp:46-87) derives from the CIGAR, in CIGAR order, with
 * read_pos already strand-flipped (ReadRec.cpp:74-75) and poly-A/T blocks removed (ReadRec.cpp:62-72).
 *   per record (32 B): ref_id, pos, mate_ref_id, mate_pos, end_pos (= GetEndPosition()),
 *                      flag (BAM FLAG), total_len (ReadRec.cpp:16-18), lowphred_run (longest run of
 *                      qualities below the -pm threshold, ReadRec.cpp:19-38), mapq, aux, blk_off
 *   per block  (12 B): ref_pos, match_ref, read_pos, match_read
 */
typedef struct sqg_batch {
    int64_t n_rec, n_blk;
    const int32_t *ref_id, *pos, *mate_ref_id, *mate_pos, *end_pos;
    const uint16_t *flag, *total_len, *lowphred_run;
    const uint8_t *mapq, *aux;
    const uint32_t *blk_off; /* n_rec + 1 entries */
    const int32_t *blk_ref_pos, *blk_match_ref;
    const uint16_t *blk_read_pos, *blk_match_read;
} sqg_batch;

/*
 * Chimeric reads after the host loader (twin of BuildChimericSBamRecord, src/ReadRec.cpp:329-413):
 * read i owns blocks [read_off[i], read_off[i+1]); the first n_first[i] of them are FirstRead, the
 * rest SecondMate, each list sorted by read position.  Block arrays are IN/OUT for
 * sqg_build_edges (LocateRead trims them in place, src/SegmentGraph.cpp:1229-1248).
 */
typedef struct sqg_chimeric {
    int64_t n_reads, n_blk;
    const uint32_t *read_off;  /* n_reads + 1 */
    const uint16_t *n_first;
    const int32_t *first_total_len, *second_total_len;
    const uint8_t *first_lowphred, *second_lowphred; /* 0/1 */
    const uint8_t *multi_filter;                      /* ReadRec_t::MultiFilter (always 0 in STAR mode) */
    int32_t *blk_ref_id, *blk_ref_pos, *blk_read_pos, *blk_match_ref, *blk_match_read;
    uint8_t *blk_is_reverse;
} sqg_chimeric;

/*
 * Replaces SegmentGraph_t::ConnectedComponent (SegmentGraph.cpp:2986-3003 with DFS :2911-2935; SURVEY.md 8f row 4) on any graph
 * given as edge end points: label[i] = index of node i's connected component, components numbered in the order of their smallest
 * node -- what the reference's repeated scan + DFS produces.  Union-find on the device (links to the smaller index) + a prefix
 * count of the roots.  Host arrays in, host array out; *n_components may be NULL.  Needs no context.
 */
int sqg_connected_components(int32_t device, int64_t n_nodes, const int32_t *ind1, const int32_t *ind2, int64_t n_edges, int32_t *label_out, int32_t *n_components);

/* Creates a context on CUDA device `device`.  ref_len[n_ref] = RefLength (ReadRec.cpp:274-279). */
int sqg_create(sqg_ctx **out, const sqg_config *cfg, const int32_t *ref_len, int32_t n_ref, int32_t device);
void sqg_destroy(sqg_ctx *ctx);
const char *sqg_last_error(const sqg_ctx *ctx);

/*
 * Replaces the three BamReader passes over the concordant BAM (SegmentGraph.cpp:293-296,
 * 1570-1577, 3126-3129): the batch is copied to HBM once and stays resident for all phases.
 * `first_record_index` is the global index of record 0 of this batch in the whole sorted stream
 * (0 on a single GPU; the shard offset when the stream is range-sharded, SURVEY.md §8e).
 */
int sqg_load_concordant(sqg_ctx *ctx, const sqg_batch *batch, int64_t first_record_index);
/*
 * Compact wire form of an sqg_batch for the host -> HBM transfer (13 B per record + 8 B per explicit block instead of 32 + 12): the
 * transfer over PCIe is what an end-to-end call waits for, so the stream is shipped delta-coded and widened on the device.
 * Records are cut into tiles of SQG_WIRE_TILE consecutive records; tile t carries the (ref_id, pos) of its first record, the
 * index of its first block in the batch (tile_blk_off) and in the wire block arrays (tile_wblk_off).  Per record: dpos = pos - pos
 * of the previous record (0 for the first record of a tile; same ref_id as that record), span = end_pos - pos, dmate = mate_pos -
 * pos (mate on the same ref_id), lowphred_run as one byte, aux (low 4 bits) | block code (high 4 bits); flag, total_len and mapq
 * are shipped as they are.  Block code 0..13 = that many explicit blocks; 14 = ONE block that the record implies (ref_pos = pos,
 * match_ref = match_read = span, read_pos = 0: an unclipped, unspliced read -- two records in three) and that is not shipped at
 * all; 15 = escape.  Per explicit block: dref = ref_pos - pos of its record and match_ref as 16 bits, read_pos, match_read.  A
 * value that does not fit is stored as the escape (0xFFFF; dmate -32768; lowphred_run 255; block code 15) and its record / block
 * is listed in full in rec_exc / blk_exc (sorted by index -- record index resp. index into the WIRE block arrays; tile t owns
 * entries [tile_rec_exc_off[t], tile_rec_exc_off[t+1]) resp. tile_blk_exc_off).  Lossless for every valid sqg_batch whose aux < 16.
 * sqh_pack_wire (squid_b200_host.h) builds it from an sqg_batch.
 */
#define SQG_WIRE_TILE 512
typedef struct sqg_wire_rec_exc { uint32_t idx; int32_t ref_id, pos, mate_ref_id, mate_pos, end_pos; uint16_t lowphred_run, n_blk; } sqg_wire_rec_exc; /* 28 B */
typedef struct sqg_wire_blk_exc { uint32_t idx; int32_t ref_pos, match_ref; } sqg_wire_blk_exc;                                                        /* 12 B */
typedef struct sqg_wire {
    int64_t n_rec, n_blk, n_tiles, n_rec_exc, n_blk_exc;
    int64_t n_wblk;                                                         /* explicit blocks = length of the wire block arrays */
    const int32_t *tile_ref_id, *tile_pos;                                  /* n_tiles */
    const uint32_t *tile_blk_off, *tile_rec_exc_off, *tile_blk_exc_off;     /* n_tiles + 1 each */
    const uint32_t *tile_wblk_off;                                          /* n_tiles + 1 */
    const uint16_t *dpos, *span; const int16_t *dmate;                      /* n_rec */
    const uint16_t *flag, *total_len; const uint8_t *lowphred_run, *mapq, *aux_nblk;
    const uint16_t *blk_dref, *blk_match_ref, *blk_read_pos, *blk_match_read; /* n_wblk */
    const sqg_wire_rec_exc *rec_exc; const sqg_wire_blk_exc *blk_exc;
} sqg_wire;
/* sqg_load_concordant() from the wire form: uploaded in record-range chunks on a copy stream, each chunk widened into the
 * resident sqg_batch layout by k_wire_decode -- and classified -- while the next ones are still in flight.  Page-locked arrays make the copies
 * asynchronous.  An inconsistent wire batch is reported (SQG_EINVAL) by the next sqg_build_nodes/sqg_build_edges/sqg_bp_coverage. */
int sqg_load_concordant_wire(sqg_ctx *ctx, const sqg_wire *wire, int64_t first_record_index);
/*
 * sqg_load_concordant() straight from the concordant BAM file (BGZF, or an uncompressed BAM stream): the compressed bytes go to
 * HBM and are inflated, cut into records and decoded there, into the same resident batch that sqh_open_bam_case packs from the
 * same file (bit-identical), so every phase after the load runs unchanged.  The inflated stream is processed in windows of whole
 * BGZF members (about 1 GiB; SQG_BAM_WINDOW_MB), so it never has to be resident as a whole.  `opt` carries the decode inputs of the
 * host packer: the quality offset and -pm threshold of the low-quality run, and ChimName (the suffix-stripped Qnames of the
 * chimeric reads and the empty name: sqh_case_chim_names of a case opened with sqh_open_bam_chimeric) as n_names names, name i =
 * names[name_off[i], name_off[i+1]); n_names = 0 probes no names.  Refusals, with the host front end's wording:
 *   SQG_EINVAL        not BGZF, no BC subfield, truncated member, member > 64 KiB, corrupt deflate stream (ISIZE mismatch
 *                     included), CRC32 mismatch, malformed header or record;
 *   SQG_EUNSUPPORTED  more than 16 blocks or TotalLen > 65535 in a record, >= 2^31 records, >= 2^32 blocks.
 * A refused load leaves no batch; the context stays usable.  Phases "bam_h2d", "bam_inflate", "bam_records", "bam_decode" (summed
 * over the windows); stats "bam_members", "bam_windows", "bam_repair_rounds".
 */
typedef struct sqg_bam_decode {
    int32_t phred33;     /* 1: qualities offset 33 (Phred_Type) */
    int32_t min_phred;   /* -pm */
    int64_t n_names;
    const char *names;
    const int64_t *name_off;  /* n_names + 1 */
} sqg_bam_decode;
int sqg_load_concordant_bam(sqg_ctx *ctx, const char *path, const sqg_bam_decode *opt, int64_t first_record_index);
/* Copies the resident batch back into caller-allocated host arrays of `out` (n_rec / n_blk must match): the check that a wire
 * upload reproduces the sqg_batch it was packed from. */
int sqg_download_concordant(sqg_ctx *ctx, sqg_batch *out);
/* Same, but the arrays of `batch` are DEVICE pointers that the caller keeps alive until sqg_destroy(). */
int sqg_attach_concordant_device(sqg_ctx *ctx, const sqg_batch *batch, int64_t first_record_index);

/* Replaces the Chimrecord argument of BuildNode_STAR/BuildEdges (SegmentGraph.cpp:192, 1932).  The arrays of `chim` must
 * stay valid and unmodified until sqg_build_nodes() or sqg_build_edges() has returned: the chimeric pre-pass
 * (SegmentGraph.cpp:196-264) reads them on a host thread while the stream works on the concordant batch. */
int sqg_load_chimeric(sqg_ctx *ctx, const sqg_chimeric *chim);

/*
 * Replaces SegmentGraph_t::BuildNode_STAR (SegmentGraph.cpp:192-831).
 * Outputs n_nodes segments tiling every chromosome, and per node three (count, sum of MatchRef)
 * pairs kept separate as the reference accumulates them: [0] discordant blocks (:773-779),
 * [1] ReadsMain (:784-801), [2] ReadsOther (:806-823); count3/sumlen3 are [3][n_nodes] int32
 * (the reference's accumulators are `int`).  `reads_other_nonempty` tells the host twin whether
 * to perform the AvgDepth division (:804, :824).
 */
int sqg_build_nodes(sqg_ctx *ctx, int32_t **chr, int32_t **pos, int32_t **len, int64_t *n_nodes,
                    int32_t **count3, int32_t **sumlen3, int32_t *reads_other_nonempty);

/* Replaces SegmentGraph_t(string graphfile)'s node reload (SegmentGraph.cpp:126-157): installs a node
 * table so that edges/coverage can run on a stored graph.  The table must tile the genome: sorted by chromosome, every
 * chromosome covered from 0 to its length by contiguous segments of positive length.  Anything else is refused with
 * SQG_EINVAL (sqg_last_error says which rule broke) and leaves the context as it was. */
int sqg_set_nodes(sqg_ctx *ctx, const int32_t *chr, const int32_t *pos, const int32_t *len, int64_t n_nodes);

/*
 * Replaces SegmentGraph_t::BuildEdges up to UpdateNodeLink (SegmentGraph.cpp:1932-1959):
 * RawEdgesChim + RawEdgesOther + sort + run-length sum + drop Weight<=0.
 * heads[i] bit0 = Head1, bit1 = Head2.  Chimeric blocks loaded by sqg_load_chimeric are trimmed
 * in place (written back into the caller's sqg_chimeric arrays passed here).
 * sqg_build_nodes() already runs the assignment pass (it shares its staging with the depth pass) and
 * caches the edge table of the segments it produced; this call then only copies it out.  After
 * sqg_set_nodes() the table is recomputed for the injected segments.
 */
int sqg_build_edges(sqg_ctx *ctx, int32_t **ind1, int32_t **ind2, uint8_t **heads, int32_t **weight, int64_t *n_edges,
                    sqg_chimeric *chim_inout);

/*
 * Replaces the BAM pass of SegmentGraph_t::ExactBPConcordantSupport (SegmentGraph.cpp:3124-3166):
 * (bp_chr, bp_pos)[n_bp] sorted by (chr, pos) as at :3109; cov_out[n_bp] = Coverages.
 */
int sqg_bp_coverage(sqg_ctx *ctx, const int32_t *bp_chr, const int32_t *bp_pos, int64_t n_bp, int32_t *cov_out);

/*
 * Multi-GPU (SURVEY.md §8e).  A range shard computes partial results; these expose them as DEVICE
 * buffers so that the caller can run the NCCL exchange and hand the merged table back.
 * (sqg_merge_edge_tables replaces the context's own table with the merged one.)
 */
int sqg_edges_device_table(sqg_ctx *ctx, uint64_t **d_keys, int32_t **d_weights, int64_t *n);
int sqg_merge_edge_tables(sqg_ctx *ctx, const uint64_t *d_keys, const int32_t *d_weights, int64_t n,
                          int32_t **ind1, int32_t **ind2, uint8_t **heads, int32_t **weight, int64_t *n_edges);

/*
 * Exact range sharding of ONE sorted stream over several contexts / GPUs (SURVEY.md 8e).  The reference has no such notion: its
 * three BamReader passes (SegmentGraph.cpp:293-296, 1570-1577, 3126-3129) walk the whole file on one thread.  Here the caller
 * cuts the stream with sqg_plan_shards(), gives every context its record range (sqg_load_concordant) and ALL chimeric reads
 * (sqg_load_chimeric), and runs the stages below, exchanging the small per-shard results between them (NCCL / torch.distributed
 * all_gather when the contexts live in different processes; squid_b200/sharded.py is that driver).  The combined outputs are
 * bit-identical to the single-context calls above.  A stream decoded on the device needs no host batch: every context loads
 * the whole stream (sqg_load_concordant_bam) and all chimeric reads, plans the same cuts on it (sqg_plan_shards_resident) and
 * keeps its own range (sqg_keep_records) -- ShardedSegmentGraph.load_bam.
 *
 *   sqg_plan_shards   cuts[0..n_planned] (cuts[0] = 0, cuts[n_planned] = n_rec); shard i owns records [cuts[i], cuts[i+1]).
 *                     Cuts are placed at coverage gaps clear of every discordant group, where BuildNode_STAR's windows are
 *                     empty and its pending segment closed (:616-636); n_planned < n_shards when the stream has too few.
 *                     All arrays of `batch` are HOST pointers.
 *   sqg_plan_shards_resident / sqg_keep_records
 *                     the same cuts from the resident batch, and one shard's range of it (see below).
 *   sqg_set_shard     declares the context shard `index` of `count` (before the stages).  Shard 0 owns the edges of the chimeric
 *                     reads and the discordant-block depth.
 *   sqg_shard_seeds   stage 1 = BuildNode_STAR up to the seed segments (:296-701) on this shard: *ops = n_ops x 4 int32
 *                     (kind, chr, pos, len) emission ops, library-owned.  prior_emission: has an earlier shard emitted an op?
 *                     (shards run with 1 speculatively; the caller repeats the stage with 0 for a shard whose predecessors all
 *                     came back empty -- until a segment exists the reference behaves differently, :545, :558).
 *   sqg_shard_build   stage 2 = the ops of ALL shards, concatenated in shard order -> segment table (:19-38, 706-761), this
 *                     shard's depth numerators (:765-826; add the count3 / sumlen3 / reads_other_nonempty of all shards) and its
 *                     edge table (sqg_edges_device_table -> all_gather -> sqg_merge_edge_tables).
 *   sqg_shard_hint_state / sqg_shard_redo_edges
 *                     LocateRead's running hint (firstfrontindex, :1568, 1612-1614) crosses shard boundaries: out_hint = the
 *                     value this shard leaves (-1: it located no read), lead_sensitive = some read of this shard depended on
 *                     the incoming value.  A shard with lead_sensitive whose true incoming hint (out_hint of the nearest
 *                     earlier shard that has one) is not the one it ran with repeats its edge pass with it.
 *   sqg_shard_cov_*   ExactBPConcordantSupport's BAM pass (:3124-3166).  begin: uploads the sorted breakpoints; *nq = this
 *                     shard's qualifying records (rank offsets = exclusive sums over the shards), *n_pass = breakpoints some
 *                     record of this shard passes.  chain: indBP enters this shard at breakpoint k_in; *k_out = first
 *                     breakpoint it leaves unresolved (= k_in of the next shard; run speculatively with k_in = max n_pass of
 *                     the earlier shards and repeat where k_out of the predecessor differs).  owned_t: writes rank_offset + t
 *                     for [k_in, k_out) into t_global[n_bp].  count: this shard's share of Coverages given the complete
 *                     t_global (unresolved breakpoints = total number of qualifying records); sum the shares.
 */
int sqg_plan_shards(const sqg_batch *batch, const sqg_chimeric *chim, const sqg_config *cfg, int32_t n_ref, int32_t n_shards,
                    int64_t *cuts, int32_t *n_planned);
/*
 * sqg_plan_shards() on the context's resident batch (any loader) and the chimeric reads of sqg_load_chimeric: cuts[0..n_planned]
 * (n_shards + 1 entries) equal to what sqg_plan_shards returns for the same stream.  The per-record part of the planner's rules
 * runs on the device on the class bytes of the classification pass (run first when the batch is not classified yet: an unsorted
 * or malformed batch is refused as there) and the discordant groups of the chimeric pre-pass; the candidates come back to the host
 * for the greedy choice of the cuts.  May be called on a context that sqg_set_shard has declared a shard.  Phase "plan".
 *   SQG_EINVAL  n_shards < 1;   SQG_ESTATE  no batch, no chimeric reads, or after sqg_keep_records.
 */
int sqg_plan_shards_resident(sqg_ctx *ctx, int32_t n_shards, int64_t *cuts, int32_t *n_planned);
/*
 * Restricts the resident batch to records [lo, hi): they become the batch (blk_off rebased to 0, block arrays from blk_off[lo]),
 * moved to the front of the context's own arrays on the device, and every product computed from the whole batch (class bytes,
 * coverage pairs, edge table) is dropped -- the context is then as if [lo, hi) had been loaded with sqg_load_concordant (with
 * first_record_index advanced by lo).  SQG_EINVAL unless 0 <= lo <= hi <= n_rec; SQG_ESTATE without a batch or when the batch is
 * attached (sqg_attach_concordant_device: caller-owned arrays).
 */
int sqg_keep_records(sqg_ctx *ctx, int64_t lo, int64_t hi);
int sqg_set_shard(sqg_ctx *ctx, int32_t index, int32_t count);
int sqg_shard_seeds(sqg_ctx *ctx, int32_t prior_emission, const int32_t **ops, int64_t *n_ops);
int sqg_shard_build(sqg_ctx *ctx, const int32_t *ops_all, int64_t n_ops_all, int32_t **chr, int32_t **pos, int32_t **len, int64_t *n_nodes,
                    int32_t **count3, int32_t **sumlen3, int32_t *reads_other_nonempty);
int sqg_shard_hint_state(sqg_ctx *ctx, int32_t *lead_sensitive, int32_t *out_hint);
int sqg_shard_redo_edges(sqg_ctx *ctx, int32_t init_hint);
int sqg_shard_cov_begin(sqg_ctx *ctx, const int32_t *bp_chr, const int32_t *bp_pos, int64_t n_bp, int64_t *nq, int64_t *n_pass);
int sqg_shard_cov_chain(sqg_ctx *ctx, int64_t k_in, int64_t *k_out);
int sqg_shard_cov_owned_t(sqg_ctx *ctx, int64_t rank_offset, int64_t k_in, int64_t k_out, int64_t *t_global);
int sqg_shard_cov_count(sqg_ctx *ctx, int64_t rank_offset, const int64_t *t_global, int32_t *cov_partial);

/* Device time in ms of the named phase/kernel of the most recent call ("classify", "seed", "tile", "depth_edges",
 * "edge_sort", "coverage", "plan"; kernels: "k_classify", "k_cov_compact", "k_assign_depth", "k_assign_edges", "k_edges_generic",
 * "k_cov_count"), measured with CUDA events on the context's stream; <0 if unknown. */
float sqg_phase_ms(const sqg_ctx *ctx, const char *name);
/* Number of kernel launches issued by this context so far. */
int64_t sqg_launch_count(const sqg_ctx *ctx);
/* Counters of the most recent calls ("islands", "heavy_islands", "groups", "disc_blocks", "gap_records", "partial_records",
 * "displaced_records", "lmax", "sensitive_reads", "raw_edges" (= (key, count) pairs before the reduce), "cov_chain_fallback",
 * "r_break", "edges_single_path", "edges_generic_path", "first_kept", "end_other", "classify_attempts"); -1 if unknown. */
int64_t sqg_stat(const sqg_ctx *ctx, const char *name);
/* Test seam of the classification pass: copies the named phase-1 array of the resident batch to `out` (classifying it first if
 * needed) and sets *n to its element count; nothing is copied when out is NULL or cap (in elements) < *n.  Names and element
 * types: "cls" (uint8, per record), "first_len" (uint16, per record), "gap_rec" (int32) and "gap_key" (uint64) for the
 * coverage-gap records, "pc_rec" and "dp_rec" (int32: partial, displaced records), per 512-record tile "okmax_excl" (uint64),
 * "ccmax" (int32), "cov_nq" (uint32), "cov_qmax" (uint64), and per record "qstage_key" (uint64), "qstage_end" (int32), compacted
 * inside each tile.  sqg_build_nodes reuses some of these buffers: call this before it. */
int sqg_classify_dump(sqg_ctx *ctx, const char *name, void *out, int64_t cap, int64_t *n);

#ifdef __cplusplus
}
#endif
#endif
