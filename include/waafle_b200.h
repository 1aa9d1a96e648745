/*
 * waafle_b200.h -- C ABI of the B200-native waafle_orgscorer engine.
 *
 * Drop-in boundary (SURVEY.md 8b).  The reference has no FFI: the boundary is a code
 * region, the body of the "major contig loop" of
 *     /root/reference/waafle/waafle_orgscorer.py:952-960
 * (Contig.attach_hits -> update_gene_scores -> [raise_taxonomy]* -> evaluate_contig) plus the
 * state it leaves for write_main_output_files (waafle_orgscorer.py:838-890: best_one /
 * best_two .ok/.crit/.rank/.clade1/.clade2/.synteny/.direction/.tails*, Locus.ignore,
 * Locus.annotations).  A maintainer replaces that block by ONE wfl_score_batch call on the
 * packed arrays below (INTEGRATION.md shows the ctypes binding).
 *
 * Conventions: plain pointers and sizes only; the caller owns every host buffer (pageable or
 * pinned); the engine owns device memory and its stream; every entry point returns 0 on
 * success and a negative wfl_status on failure and never throws / aborts; wfl_last_error()
 * gives the text.  One handle per GPU; a handle is not thread-safe, distinct handles are
 * independent.  There is no CPU fallback: without a CUDA device wfl_create fails.
 */
#ifndef WAAFLE_B200_H
#define WAAFLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WFL_ABI_VERSION 2
#define WFL_MAX_SYSTEMS 32

typedef struct wfl_engine wfl_engine;

typedef enum {
    WFL_OK = 0,
    WFL_ERR_ARG = -1,       /* bad argument / inconsistent batch            */
    WFL_ERR_CUDA = -2,      /* CUDA runtime error (text in wfl_last_error)   */
    WFL_ERR_STATE = -3,     /* params / taxonomy / batch not set             */
    WFL_ERR_CAPACITY = -4,  /* caller-provided output buffer too small       */
    WFL_ERR_RUNAWAY = -5,   /* >100 taxonomy lifts (reference: wu.die, waafle_orgscorer.py:580-581) */
    WFL_ERR_RANGE = -6,     /* a score outside the range the details formatter prints exactly (|x| < 2^53)  */
    WFL_ERR_DATA = -7       /* compressed input that fails validation (wfl_inflate_bgzf)  */
} wfl_status;

/* Engine-relevant CLI flags (waafle_orgscorer.py:188-296, waafle_genecaller.py:83-101;
 * read inside the engine at waafle_orgscorer.py:338-346,351,362,365,367,413-420,497,
 * 513-516,589,604,610,625-627,636,644-661,679-687,701,707,714,720-721,741). */
typedef struct {
    double k1;                    /* --one-clade-threshold                      */
    double k2;                    /* --two-clade-threshold                      */
    double range;                 /* --range                                    */
    double ambiguous_fraction;    /* --ambiguous-fraction                       */
    double min_overlap;           /* --min-overlap                              */
    double min_scov;              /* --min-scov                                 */
    double min_gene_length;       /* --min-gene-length                          */
    int32_t disambiguate_one;     /* 0 report-best, 1 meld                      */
    int32_t disambiguate_two;     /* 0 report-best, 1 jump, 2 meld              */
    int32_t weak_loci;            /* 0 ignore, 1 penalize, 2 assign-unknown     */
    int32_t ambiguous_threshold;  /* 0 off, 1 lenient, 2 strict                 */
    int32_t sister_penalty;       /* 0 off, 1 lenient, 2 strict                 */
    int32_t annotation_threshold; /* 0 off, 1 lenient, 2 strict                 */
    int32_t allow_lca;            /* --allow-lca                                */
    int32_t stranded;             /* --stranded                                 */
    int32_t jump_taxonomy;        /* --jump-taxonomy, 0 = off                   */
    int32_t clade_genes;          /* --clade-genes, -1 = off                    */
    int32_t clade_leaves;         /* --clade-leaves, -1 = off                   */
    int32_t n_systems;            /* annotation systems carried by hit_sysmask  */
} wfl_params;

/* One batch of contigs, CSR over contigs, SoA over hits and loci.
 * Replaces the per-contig Hit / Locus object lists (waafle/utils.py:192-241, 298-322).
 * Contigs in FASTA order, loci in GFF order (ALL loci; the engine applies
 * --min-gene-length, waafle_orgscorer.py:350-352), hits in blastout order. */
typedef struct {
    int64_t n_contigs, n_hits, n_loci;
    const int64_t *hit_off;        /* [n_contigs+1] */
    const int64_t *locus_off;      /* [n_contigs+1] */
    const int32_t *hit_qstart;     /* [n_hits] Hit.qstart                                */
    const int32_t *hit_qend;       /* [n_hits] Hit.qend                                  */
    const int32_t *hit_taxon;      /* [n_hits] node index of Hit.taxon                   */
    const double  *hit_score;      /* [n_hits] Hit.waafle_score   (utils.py:229)         */
    const double  *hit_scov;       /* [n_hits] Hit.scov_modified  (utils.py:227)         */
    const int8_t  *hit_strand;     /* [n_hits] '+' or '-'         (utils.py:214)         */
    const uint32_t *hit_sysmask;   /* [n_hits] bit s: hit annotates system s; NULL if n_systems==0 */
    const int32_t *locus_start;    /* [n_loci] */
    const int32_t *locus_end;      /* [n_loci] */
    const int8_t  *locus_strand;   /* [n_loci] first byte of the GFF strand column */
} wfl_batch;

/* The same batch in the COMPACT wire format: 14 bytes per hit instead of 29 (the plugin call is bound by the
 * host->device link).  What is dropped is what the engine does not need per hit: scov_modified is used for exactly
 * one comparison (waafle_orgscorer.py:362), which the host applies while packing (utils.py:214-229 already computes
 * the value) and ships as one bit; the strand is one bit (utils.py:214); node indices and query coordinates fit 14 and
 * 16 bits.  Usable when the taxonomy has <= 16384 nodes, every query coordinate is <= 65535 and n_systems <= 8
 * (the engine rejects the batch otherwise).  Results are identical to the wide format's. */
typedef struct {
    int64_t n_contigs, n_hits, n_loci;
    const int64_t *hit_off;        /* [n_contigs+1] */
    const int64_t *locus_off;      /* [n_contigs+1] */
    const uint16_t *hit_qstart16;  /* [n_hits] Hit.qstart                                              */
    const uint16_t *hit_qend16;    /* [n_hits] Hit.qend                                                */
    const uint16_t *hit_tax16;     /* [n_hits] bits 0-13 node index of Hit.taxon, bit 14 sstrand == '-',
                                      bit 15 scov_modified >= --min-scov                              */
    const double   *hit_score;     /* [n_hits] Hit.waafle_score                                        */
    const uint8_t  *hit_sysmask8;  /* [n_hits] bit s: hit annotates system s; NULL if n_systems == 0   */
    const int32_t *locus_start;    /* [n_loci] */
    const int32_t *locus_end;      /* [n_loci] */
    const int8_t  *locus_strand;   /* [n_loci] */
} wfl_packed_batch;
#define WFL_PACKED_MAX_NODES 16384
#define WFL_PACKED_MAX_COORD 65535
#define WFL_PACKED_MAX_SYSTEMS 8

/* call codes */
#define WFL_CALL_UNCLASSIFIED 0
#define WFL_CALL_NO_LGT 1
#define WFL_CALL_LGT 2
/* locus_flags bits */
#define WFL_LOCUS_RETAINED 1
#define WFL_LOCUS_IGNORED 2

/* Caller-allocated result buffers (capacities in elements; sizes returned in *_used).
 * Replaces Contig.best_one / best_two, Locus.ignore and Locus.annotations. */
typedef struct {
    /* per contig [n_contigs] */
    uint8_t *call;          /* WFL_CALL_*                                               */
    uint8_t *direction;     /* 0 "A?B", 1 "B>A"       (waafle_orgscorer.py:485,543)     */
    int32_t *lifts;         /* taxonomy lifts performed (jumps + loop)                  */
    int32_t *clade1;        /* clade / clade_A after melding, -1 if unclassified        */
    int32_t *clade2;        /* clade_B after melding, -1 unless lgt                     */
    int32_t *lca;           /* LCA(clade_A, clade_B), -1 unless lgt                     */
    int32_t *best1;         /* clade1 of the best option before melding                 */
    int32_t *best2;
    double  *crit;          /* min_score / min_max_score                                */
    double  *rank;          /* avg_score / avg_max_score                                */
    int64_t *member_off;    /* [n_contigs+1] CSR into members                           */
    int32_t *n_members_a;   /* first n_members_a of a contig's members are side A       */
    /* distinct melded clades (tails are derived on the host, waafle_orgscorer.py:750-759) */
    int32_t *members;
    int64_t members_capacity;
    int64_t members_used;   /* out */
    /* per raw locus [n_loci] */
    uint8_t *synteny;       /* synteny character, 0 for dropped loci / unclassified     */
    uint8_t *locus_flags;   /* WFL_LOCUS_*                                              */
    int32_t *ann_winner;    /* [n_loci * n_systems] batch hit index or -1               */
    /* on-device compaction: contig indices grouped lgt | no_lgt | unclassified */
    int64_t *call_counts;   /* [3] = {n_lgt, n_no_lgt, n_unclassified}                  */
    int64_t *call_index;    /* [n_contigs]                                              */
} wfl_results;

/* Counters of the last run (metrics / bench evidence). */
typedef struct {
    int64_t kernel_launches;    /* kernels launched by the last score/run call           */
    int64_t contigs, hits, loci;
    int64_t matched_pairs;      /* (hit, locus) matches                                  */
    int64_t groups;             /* (clade, locus) envelopes integrated, all levels       */
    int64_t levels;             /* sum over contigs of taxonomy levels evaluated         */
    int64_t pairs_tested;       /* two-clade pairs mask-tested                           */
    int64_t pairs_scored;       /* two-clade pairs that passed the mask test             */
    int64_t workspace_retries;  /* contigs replayed by the exact pipeline with a larger workspace */
    int64_t smem_contigs;       /* contigs scored entirely in shared memory by the fused fast-path kernel */
    int64_t fallback_contigs;   /* contigs the fast path handed to the exact pipeline (capacity or guard band) */
    int64_t second_pass_contigs;/* contigs the first fast pass handed to a retry pass (more survivor pairs / larger slice) */
    int64_t fallback_reasons[8];/* hand-overs of both passes by cause: loci, hits, coordinates, records, clades,
                                   groups, pairs, guard band */
    int64_t guard_trips;        /* ... of which because a rank comparison fell inside the 1e-12 guard band */
    int64_t refined_groups;     /* gene scores recomputed in numpy's summation order inside the fast kernel */
    int64_t host_syncs;         /* stream synchronisations inside the last call          */
    int64_t phase_cycles[12];   /* per-phase SM cycles of the exact pipeline (only with -DWFL_PROFILE) */
    float   ms_h2d, ms_kernels, ms_d2h, ms_score_kernel;   /* CUDA-event times         */
} wfl_stats;

int  wfl_abi_version(void);
int  wfl_device_count(void);
int  wfl_create(int device, wfl_engine **out);
void wfl_destroy(wfl_engine *e);
const char *wfl_last_error(const wfl_engine *e);

int  wfl_set_params(wfl_engine *e, const wfl_params *p);
/* Node index order must equal the Python str order of the clade names (so that
 * `clade1 < clade2`, waafle_orgscorer.py:608, is an integer compare).  parent[root] == root;
 * unlisted taxa have parent == root (utils.py:386-387), listed == 0, leaf_count == 1. */
int  wfl_set_taxonomy(wfl_engine *e, int32_t n_nodes, const int32_t *parent,
                      const int32_t *depth, const int32_t *leaf_count, const uint8_t *listed,
                      int32_t root_idx, int32_t unknown_idx);

/* Host buffers in, host buffers out: H2D + kernels + D2H (the plugin call; bench "e2e").  `out` may be NULL: the
 * results then stay on the device (wfl_pack_results / wfl_download_results fetch them). */
int  wfl_score_batch(wfl_engine *e, const wfl_batch *in, wfl_results *out);
int  wfl_score_packed(wfl_engine *e, const wfl_packed_batch *in, wfl_results *out);

/* Split form for device-resident timing (bench "value"): upload once, run many, download. */
int  wfl_upload_batch(wfl_engine *e, const wfl_batch *in);
int  wfl_upload_packed(wfl_engine *e, const wfl_packed_batch *in);
int  wfl_run_resident(wfl_engine *e);
int  wfl_download_results(wfl_engine *e, wfl_results *out);

int  wfl_get_stats(const wfl_engine *e, wfl_stats *out);
/* Tuning / test knobs by name (all optional; defaults are the measured best on B200):
 *   "exact"        1: every contig through the exact pipeline (numpy-pairwise gene scores, bit-exact crit / rank);
 *                  0 (default): fused fast-path kernel with guard bands, exact pipeline for what it hands back
 *   "fast_hcap" / "fast_tcap" / "fast_ncap"   capacities of the fast kernel's shared-memory slice (staged hit x locus
 *                  entries per contig, clades and groups per level); 0 = choose from the batch;
 *                  "fast_hscale_pct" first-pass entry capacity in % of the mean hits per contig (default 160);
 *                  "fast_passes" 1: no retry passes (overflows go straight to the exact pipeline)
 *   "details"      capacity of the --write-details dump (wfl_download_details); > 0 implies the exact pipeline
 *   "pool_mb"      workspace pool of the exact pipeline; "chunk_mb" H2D chunk of the plugin call; "streams" 1|2;
 *   "k2_cap"       group-list capacity of the exact pipeline (test hook for its overflow path). */
int  wfl_set_option(wfl_engine *e, const char *name, int64_t value);

/* Multi-GPU gather support (SURVEY 8e): the compacted results of the last run, packed by one kernel into ONE
 * device buffer on the engine's stream, ready for a single NCCL gather.  Layout: 8 int64 header {n_contigs, n_loci,
 * n_systems, n_members, 0...}, then the wfl_results arrays in declaration order, each section 16-byte aligned
 * (wfl_packed_results_layout gives the offsets for given sizes).  The pointer stays valid until the next call on
 * this engine; `stream` is the cudaStream_t the buffer is ordered on. */
int  wfl_pack_results(wfl_engine *e, void **dev_ptr, int64_t *bytes, void **stream);
/* byte offsets of the 18 sections {call, direction, lifts, clade1, clade2, lca, best1, best2, crit, rank, member_off,
 * n_members_a, members, synteny, locus_flags, ann_winner, call_counts, call_index} and the total size */
int64_t wfl_packed_results_layout(int64_t n_contigs, int64_t n_loci, int32_t n_systems, int64_t n_members,
                                  int64_t offsets[18]);

/* ---- front end on the device (SURVEY 8f rank 1): BLAST outfmt-6 text -> hit columns -------------------------------
 * Replaces the per-row Hit objects of waafle/utils.py:192-241 / iter_contig_hits :255-270.  The caller ships the raw
 * text of a blastout file; the device splits rows and fields, converts the numbers exactly, computes scov_modified and
 * waafle_score in the reference's operation order (utils.py:214-229), dictionary-codes the taxon (sseqid field 1) and
 * the annotation systems (fields 2+) against hash sets of the file's DISTINCT names, and flags contig block starts.
 * Rows it cannot reproduce exactly are counted in *flagged: the caller must then use its CPU reader. */
typedef struct wfl_parser wfl_parser;
int  wfl_parser_create(int device, wfl_parser **out);
void wfl_parser_destroy(wfl_parser *p);
const char *wfl_parser_last_error(const wfl_parser *p);
/* returns the number of rows or a negative wfl_status; = an upload of the text followed by wfl_parse_blast_resident */
int64_t wfl_parse_blast(wfl_parser *p, const char *text, int64_t n_bytes, int32_t *flagged, int64_t *first_flagged);
/* Parse bytes [off, off + n_bytes) of the text already resident on the parser (the last wfl_parse_blast upload or
 * wfl_inflate_bgzf).  Same results as wfl_parse_blast on those bytes: ss_off / q_off and the distinct-name offsets are
 * relative to `off`.  WFL_ERR_ARG for a range outside the resident text. */
int64_t wfl_parse_blast_resident(wfl_parser *p, int64_t off, int64_t n_bytes, int32_t *flagged, int64_t *first_flagged);
/* Copy resident text [off, off + n_bytes) to dst (the host side's names are slices of it). */
int  wfl_parser_text(wfl_parser *p, int64_t off, int64_t n_bytes, char *dst);
/* BGZF (bgzip's gzip variant) inflated on the device into the parser's resident text.  `comp`: the compressed bytes;
 * `members`: [n_members][5] = offset of the raw DEFLATE payload in comp, its length, ISIZE, CRC-32 and the member's
 * output offset (an exclusive prefix sum of ISIZE; members of at most 64 KB).  Every member is decoded and checked
 * (stored / fixed / dynamic blocks; bounds of the payload, code-length sets, symbols 286-287 and distances 30-31, no
 * distance before the member's start, exactly ISIZE bytes, the CRC-32).  Returns the text length; WFL_ERR_DATA when a
 * member fails (*bad_member = the first one, else -1: the caller reads the file on the host), WFL_ERR_ARG for a member
 * table that does not fit `comp` or does not tile the text.  ms_* (NULL = skip): CUDA-event times of the upload and of
 * the inflate kernel. */
int64_t wfl_inflate_bgzf(wfl_parser *p, const uint8_t *comp, int64_t comp_len, const int64_t *members, int64_t n_members,
                         int64_t *bad_member, float *ms_h2d, float *ms_kernel);
/* distinct-name sets of the last parse: kind 0 = taxa (2^20 slots), 1 = annotation systems (64 slots); hash[s] != 0 marks
 * an occupied slot and (off[s], len[s]) is one occurrence of its name in the text */
int  wfl_parse_distinct(wfl_parser *p, int kind, uint64_t *hash, int64_t *off, int32_t *len, int32_t slots);
/* sys_perm[slot] = bit of that system in the sorted system list (-1 for empty slots); columns of [n_rows] each, NULL = skip;
 * tcode[r] = slot of the row's taxon in the distinct-taxon set; newblock[r] = qseqid differs from the previous row's */
int  wfl_parse_fetch(wfl_parser *p, const int32_t *sys_perm, int32_t *qstart, int32_t *qend, double *score, double *scov,
                     int8_t *strand, int32_t *tcode, uint32_t *sysmask, int64_t *ss_off, int32_t *ss_len, uint8_t *newblock,
                     int64_t *q_off, int32_t *q_len);
int  wfl_parser_times(const wfl_parser *p, float *ms_h2d, float *ms_kernels, float *ms_d2h);
/* GFF text -> locus columns (replaces the per-row Locus objects of waafle/utils.py:298-355 / iter_contig_loci :341-355):
 * returns the number of TEXT rows; comment ('#') and empty rows come back with skip = 1.  newblock[r] = the seqname differs
 * from the previous locus row's; (s_off, s_len) = the seqname in the text.  *flagged rows (field count != 9, non-integer
 * coordinates, a quoted field, a strand that is not one character) send the caller to its CPU reader. */
int64_t wfl_parse_gff(wfl_parser *p, const char *text, int64_t n_bytes, int32_t *flagged, int64_t *first_flagged);
int  wfl_parse_gff_fetch(wfl_parser *p, int32_t *start, int32_t *end, int8_t *strand, uint8_t *skip, uint8_t *newblock,
                         int64_t *s_off, int32_t *s_len);
/* Gene calls (waafle_genecaller.py:107-170, as wfl_call_genes below) over the hit columns of the last successful
 * wfl_parse_blast on this parser: no hit data is re-uploaded.  keep = (scov_modified >= min_scov) on the parser's own
 * doubles; contig blocks are the parser's newblock runs, in file order.  Returns the number of genes (>= 0) or a negative
 * wfl_status: WFL_ERR_STATE when no blastout was parsed or the last parse flagged rows.  *n_blocks receives the block count
 * (an empty blastout: 0 blocks, 0 genes); *ms_kernel the device time.  A wfl_parse_gff on the same handle keeps the blast
 * columns (it parses into columns of its own), so gene calls may follow it. */
int64_t wfl_parser_call_genes(wfl_parser *p, double min_overlap, double min_gene_length, double min_scov,
                              int64_t *n_blocks, float *ms_kernel);
/* The genes of the last wfl_parser_call_genes as a dense CSR over blocks: gene_off[n_blocks+1], start / end / strand
 * [n_genes] (strand: '+' / '-').  WFL_ERR_STATE before any gene call since the last wfl_parse_blast. */
int  wfl_parser_genes_fetch(wfl_parser *p, int64_t *gene_off, int32_t *start, int32_t *end, int8_t *strand);

/* ---- the scoring batch built from a parser's resident hit columns ----------------------------------------------------
 * The wide wfl_batch of the parser's last wfl_parse_blast / wfl_parse_blast_resident, built in the engine's input
 * buffers without the hit columns crossing PCIe.  Contig c takes parser rows [hit_src[c], hit_src[c] + hit_off[c+1] -
 * hit_off[c]) (one blastout block); the taxon becomes slot_node[slot of the row's taxon] (the slots of
 * wfl_parse_distinct kind 0); the annotation systems are re-ordered through sys_perm as wfl_parse_fetch does.  Without
 * annotation systems (n_systems == 0) every contig's hits are ordered as Batch.sort_hits (waafle_b200/packing.py) orders
 * them on the host, so the batch is byte for byte the one the host packer would upload.  Loci and offsets come from
 * the host as in wfl_batch. */
typedef struct {
    int64_t n_contigs, n_hits, n_loci;
    const int64_t *hit_off;        /* [n_contigs+1] host */
    const int64_t *hit_src;        /* [n_contigs]  first parser row of contig c's block */
    const int32_t *slot_node;      /* [2^20] distinct-taxon slot -> node index, -1 unused */
    const int32_t *sys_perm;       /* [64] as wfl_parse_fetch; NULL when n_systems == 0 */
    const int64_t *locus_off; const int32_t *locus_start, *locus_end; const int8_t *locus_strand;
} wfl_parsed_batch;
/* Leaves a resident batch that wfl_run_resident, wfl_download_results, wfl_pack_results and wfl_details_* use exactly
 * like one from wfl_upload_batch.  The engine's stream waits for the parser's stream; the call returns when the batch is
 * in place (*ms_kernels, NULL = skip: device time of the gather and sort kernels).  Errors, after which the engine has no
 * batch: WFL_ERR_STATE when the parser's last parse flagged rows (or none was made) or params / taxonomy are missing;
 * WFL_ERR_ARG when the parser is on another device, offsets do not span or are not monotone, a contig's row range lies
 * outside the parser's rows, a hit's slot maps to -1 or to a node >= n_nodes, or sys_perm is NULL with n_systems > 0
 * or given with n_systems == 0. */
int  wfl_upload_parsed(wfl_engine *e, const wfl_parser *p, const wfl_parsed_batch *in, float *ms_kernels);
/* Test hook: the hit columns of the resident wide batch to the host (each [n_hits], NULL = skip; sysmask only with
 * n_systems > 0).  WFL_ERR_STATE without a resident wide batch. */
int  wfl_debug_resident_batch(wfl_engine *e, int32_t *qstart, int32_t *qend, int32_t *taxon, double *score,
                              double *scov, int8_t *strand, uint32_t *sysmask);

/* ---- --write-details (waafle_orgscorer.py:766-812) -----------------------------------------------------------------
 * With the option "details" = <capacity> set (wfl_set_option) every run goes through the exact pipeline and records, per
 * contig and evaluated taxonomy level, every gene score of every clade (write_details :802-812 walks contig.gene_scores):
 * entry = (contig index, evaluation index 0,1,2,..., clade node index, locus index within the contig (GFF order), score).
 * Scores absent from the dump are 0 (a clade has no hit on that locus, :404-405).  wfl_download_details copies up to
 * `capacity` entries (any order; a replayed contig may appear twice with identical values) and returns the number the run
 * produced. */
int64_t wfl_download_details(wfl_engine *e, int32_t *contig, int32_t *iteration, int32_t *clade, int32_t *locus, double *score,
                             int64_t capacity);
/* The details table as text, built on the device from the dump of the last run:
 *     contig \t iteration \t clade \t gene_scores \t gene_spans \n
 * per contig (in the caller's order), evaluated level (iteration = max(1, evaluation index)) and clade (ascending node
 * index), scores printed like Python's "{:.3f}", spans as write_details (:773-791) derives them from the site arrays.
 * wfl_set_clade_names: the names of the taxonomy's nodes, name i = blob[off[i], off[i+1]); once per wfl_set_taxonomy.
 * wfl_details_prepare: `order` lists n_order distinct contig indices of the batch (contigs not listed, and contigs that
 * were never evaluated, have no rows); contig c is named names[names_off[c], names_off[c+1]).  Returns the table's size
 * in bytes; bytes_before[r] (n_order + 1 entries, NULL = skip) = bytes of the rows of order[0, r).  Errors: WFL_ERR_STATE
 * without a details run or without clade names, WFL_ERR_CAPACITY when the dump overflowed its capacity, WFL_ERR_RANGE
 * when a score cannot be printed exactly.
 * wfl_details_text: the rows of order[r0, r1); returns their size and writes them to `buf` when capacity >= size (so a
 * large table is fetched in bounded pieces).  WFL_ERR_STATE without a prepare since the last run.
 * ms_* (NULL = skip): CUDA-event times of the text kernels and of the copy to `buf`. */
int  wfl_set_clade_names(wfl_engine *e, int32_t n_nodes, const char *blob, const int64_t *off);
int64_t wfl_details_prepare(wfl_engine *e, int64_t n_order, const int32_t *order, const char *names, const int64_t *names_off,
                            int64_t *bytes_before, float *ms_kernels);
int64_t wfl_details_text(wfl_engine *e, int64_t r0, int64_t r1, char *buf, int64_t capacity, float *ms_kernels,
                         float *ms_d2h);

/* ---- waafle_genecaller on the device (SURVEY 8f): gene calls from BLAST hits ------------------------------------
 * Replaces the per-contig body of waafle/waafle_genecaller.py:207-230 (hits2ints :107-113, overlap_intervals :137-168,
 * merge_inodes :121-135 over INode / calc_overlap, waafle/utils.py:455-500).  Contig blocks are consecutive runs of one
 * query in the blastout (iter_contig_hits, utils.py:255-270): hits [block_off[b], block_off[b+1]).  keep[h] = the hit passed
 * --min-scov.  The genes of block b come back at [block_off[b], block_off[b] + gene_count[b]) of the gene arrays (each as
 * long as the hit arrays), in the reference's output order.  `--stranded` has no effect upstream (:215 compares a bool with
 * "on") and is therefore not a parameter.  Host pointers in and out; returns a wfl_status. */
int  wfl_call_genes(int device, int64_t n_blocks, const int64_t *block_off, const int32_t *qstart, const int32_t *qend,
                    const int8_t *strand, const uint8_t *keep, double min_overlap, double min_gene_length,
                    int32_t *gene_start, int32_t *gene_end, int8_t *gene_strand, int32_t *gene_count, float *ms_kernel);

/* Page-locked host memory for callers without a CUDA binding of their own (pinned buffers make the
 * H2D / D2H copies of wfl_score_batch asynchronous and ~2x faster).  Free with wfl_host_free. */
int  wfl_host_alloc(size_t bytes, void **out);
void wfl_host_free(void *p);

/* Test hook: level-0 gene scores of one contig of the resident batch as COO triples
 * (clade, retained-locus index, score); returns the number of triples or <0. */
int64_t wfl_debug_gene_scores(wfl_engine *e, int64_t contig, int32_t *clade, int32_t *locus,
                              double *score, int64_t capacity);
/* Test hook: x[i] printed by the details table's "{:.3f}" formatter into text[24 i, 24 i + len[i]); returns n, or
 * WFL_ERR_RANGE if some x[i] lies outside |x| < 2^53 (len[i] = -1 there). */
int64_t wfl_debug_format_scores(wfl_engine *e, const double *x, int64_t n, char *text, int32_t *len);

#ifdef __cplusplus
}
#endif
#endif /* WAAFLE_B200_H */
