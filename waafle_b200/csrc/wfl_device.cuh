// Device-side data structures shared by the kernels and the C-ABI host code.
// Hand-written for sm_100a; no library kernels on the path.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "waafle_b200.h"

namespace wfl {

// Read-only taxonomy tables (host flattening of waafle/utils.py:374-447).
struct DevTax {
    const int32_t *parent;
    const int32_t *depth;
    const int32_t *leaf_count;
    const uint8_t *listed;
    int32_t n_nodes, root, unknown;
};

// The resident batch (wfl_batch with device pointers).
struct DevBatch {
    int64_t n_contigs, n_hits, n_loci;
    const int64_t *hit_off, *locus_off;
    const int32_t *hit_qstart, *hit_qend, *hit_taxon;
    const double *hit_score, *hit_scov;
    const int8_t *hit_strand;
    const uint32_t *hit_sysmask;
    const int32_t *locus_start, *locus_end;
    const int8_t *locus_strand;
    // compact wire format (wfl_packed_batch): 14 B/hit; null in the wide format
    const uint16_t *hit_qstart16, *hit_qend16, *hit_tax16;
    const uint8_t *hit_sysmask8;
};

// Result arrays on the device (wfl_results) plus the member staging pool.
struct DevOut {
    uint8_t *call, *direction;
    int32_t *lifts, *clade1, *clade2, *lca, *best1, *best2;
    double *crit, *rank;
    uint8_t *synteny, *locus_flags;
    int32_t *ann_winner;
    // members are bump-allocated in a staging pool by the scoring kernel, then compacted
    // into contig order (CSR) by the compaction kernels
    int32_t *n_mem_a, *n_mem_b;
    int64_t *mem_pos;
    int32_t *mem_pool;
    int64_t mem_pool_cap;
    uint8_t *status;          // per contig: 0 ok, 1 workspace overflow (replay), 2 runaway, 3 bad input
};

// Global counters (one struct in device memory, zeroed before each run).
struct DevCounters {
    unsigned long long next_work;       // work-queue head
    unsigned long long mem_pool_used;   // staging pool bump pointer (may exceed capacity)
    unsigned long long n_overflow;      // contigs that overflowed their workspace (status 1: replayed)
    unsigned long long n_runaway;
    unsigned long long n_badinput;      // contigs with a taxon index outside the taxonomy
    unsigned long long matched_pairs, groups, levels, pairs_tested, pairs_scored, smem_contigs;
    unsigned long long n_fallback;      // contigs the first fast-path pass handed on (to the second pass)
    unsigned long long n_fallback_pairs;   // contigs of the first pass whose two-clade survivor list overflowed (pairs pass)
    unsigned long long n_fallback2;     // contigs the last pass (larger slice) handed to the exact pipeline
    unsigned long long fb_reason[8];    // why (both passes): loci, hits, coordinates, records, clades, groups, pairs, guard
    unsigned long long guard_trips;     // ... of which because a rank comparison fell inside the guard band
    unsigned long long refined_groups;  // gene scores recomputed exactly inside the fast kernel (near a threshold)
    unsigned long long phase_cycles[12];   // thread-0 clock64 deltas per phase (profiling aid)
};

// Thresholds derived once on the host (waafle_orgscorer.py:338-346, 515-516, 720-721).
struct DevParams {
    wfl_params p;
    double min_thr, max_thr, ann_thr, k_amb, sister_thr;
    int amb_sel, sis_sel;     // which of the three per-clade masks (0:k1 1:k2 2:eps) to use
};

// Leaf plan of numpy's pairwise sum over n elements: data[off .. off+nleaf) holds
// (leaf size m) | (number of pending left sums to add after the leaf) << 8; k8 packs up to four
// distinct m/8 values (ascending, 0 = unused / memo disabled).
struct PlanEntry {
    uint32_t off, nleaf, k8;
};

// ---- fused fast-path kernel (wfl_fast.cu) ---------------------------------------------------
// Layout of one warp's shared-memory slice (byte offsets) and its capacities; computed on the host.
struct FastCfg {
    int slice_bytes;
    int Hcap;      // staged entries of one contig: one per (hit, locus) match == record; hits matching no locus are dropped
    int Pcap;      // power of two >= Hcap: the permutation of the per-level hit sort
    int Mcap;      // records (hit x locus matches) of one contig
    int Tcap;      // distinct clades per level
    int Ncap;      // (clade, locus) groups per level
    int Scap;      // two-clade pairs that pass the mask prefilter
    int x_bytes;   // search scratch (aliases the per-level record / group arrays, dead by then)
    int scratch_bytes;   // global scratch per resident warp: locus masks of the staged hits + cold-path record arrays
    int o_stat, o_llo, o_llen, o_lraw, o_lstr, o_lbase, o_lcur, o_llast, o_maxb, o_unk;
    int o_hv, o_hsp, o_hcl, o_hid, o_hloc;
    int o_rec, o_gstart, o_gt, o_gloc, o_x;
    int o_row;     // gene scores in clade-major CSR order
    int o_hp;      // sort permutation of the entries (u16[Pcap])
    int sort_bytes;   // bytes from o_x to the end of the rows: key array of the per-level sort
    int o_clid, o_mk0, o_mk1, o_mk2, o_pres, o_cstart;
};

struct FastArgs {
    DevBatch b;
    DevTax t;
    DevOut o;
    DevParams P;
    DevCounters *ctr;
    FastCfg cfg;
    unsigned long long *wq;        // work-queue head of this launch
    int64_t n_work, work_base;     // contig range ...
    const int *work_list;          // ... or explicit list, whose length may live on the device:
    const unsigned long long *n_work_dev;   // (second pass: the first pass's fallback count)
    int *fb_list;                  // contigs that overflowed a capacity of this pass's slice (next pass) ...
    unsigned long long *fb_count;  // ... and their number
    int *fb_pairs;                 // contigs whose ONLY problem is the survivor-pair capacity (same slice, larger Scap) ...
    unsigned long long *fb_pairs_count;   // ... null: they go to fb_list like the other overflows
    int *fb_final;                 // contigs for the exact pipeline (guard band, > 32 loci, long genes, ...)
    unsigned long long *fb_final_count;
    const int *anc;                // [anc_rows][n_nodes]: l-th ancestor of every node (row 0 = identity)
    int anc_rows;
    double guard;                  // guard band of the decision compares (1e-12)
    int qbits;                     // score bits in the keys of the per-level sort: 48 - bits(n_nodes), at most 32
    int plan_nmax;
    const PlanEntry *plan_index;
    const uint16_t *plan_data;
    char *scratch;                 // cfg.scratch_bytes per resident warp
};
int fast_layout(FastCfg &F, int Hcap, int Mcap, int Tcap, int Ncap, int Scap, int n_systems);
int fast_warps_per_cta();
int fast_ctas_per_sm(const FastCfg &F, bool packed, size_t smem_per_sm);
cudaError_t launch_fast(const FastArgs &a, bool packed, int grid, cudaStream_t s);

// ---- multi-kernel pipeline (wfl_pipeline.cu) ------------------------------------------------
enum { PIPE_DONE = 0, PIPE_ACTIVE = 1 };

// Per-contig context carried between the pipeline kernels.
struct PipeCtg {
    unsigned long long offA, offB, offC;   // workspace regions in the pool (loci | records+table | level)
    unsigned int capA, capB, capC;
    int G, W, M, T, np_tot, lifts, iter;
    int Ngrp, ng, nlt, nu, t_unk, nun, hasroot;   // written by the scores kernel for the search kernels
    int state;
};

// One (clade, locus) group of one contig as a self-contained K2 work item (64 bytes): the regroup kernel emits
// them into a per-sub-batch list, a counting sort by (leaf count, record-count class) orders them, and the K2
// kernel walks the list lane per group, so that the 32 lanes of a warp follow the same leaf plan.
struct K2Desc {
    const int *sa;                 // slice starts of the contig's records in group order; ends at sa + d_sb
    const uint16_t *plan;          // leaf plan of the gene length
    double *out;                   // g_score slot
    unsigned long long *maxb;      // per-locus max (order-preserving bits); null for the Unknown clade
    int d_sb, d_sv;                // sb = sa + d_sb (ints); sv = (double *)((char *)sa + d_sv)
    int rs, re, n, nleaf;
    unsigned int k8;
    unsigned int key;
};
constexpr int K2_KEYS = 512;       // (min(nleaf, 127) << 2) | record-count class
struct K2Meta {                    // one per taxonomy level, zeroed per sub-batch
    unsigned int hist[K2_KEYS];
    unsigned int cursor[K2_KEYS];
    unsigned long long count, take;
};

struct PipeArgs {
    DevBatch b;
    DevTax t;
    DevOut o;
    DevParams P;
    DevCounters *ctr;
    unsigned long long *wq;        // work-queue head of THIS launch
    int64_t n_work, work_base;     // prepare: contig range of the sub-batch ...
    const int *work_list;          // ... or an explicit list of n_work contig indices (replays, fast-path fallbacks)
    char *pool;                    // workspace pool of the sub-batch
    unsigned long long *pool_used;
    unsigned long long pool_cap;
    PipeCtg *ctg;                  // [n_contigs]
    int *list_act, *list_two, *list_next, *list_lift;   // device work lists (contig indices)
    int *cnt_act, *cnt_two, *cnt_next, *cnt_lift;
    int plan_nmax;
    const PlanEntry *plan_index;
    const uint16_t *plan_data;
    K2Desc *k2_desc;
    unsigned int *k2_order;
    unsigned int *k2_keys;         // sort key of every descriptor (compact copy for the counting sort)
    unsigned long long k2_cap;
    K2Meta *k2_meta;               // this level's
    // --write-details (waafle_orgscorer.py:802-812): every gene score of every clade, per contig and evaluated level
    unsigned long long *det_count;
    long long det_cap;
    int32_t *det_contig, *det_iter, *det_clade, *det_locus;
    double *det_score;
    long long dbg_contig;
    int32_t *dbg_clade, *dbg_locus;
    double *dbg_score;
    long long dbg_cap;
    long long *dbg_count;
};

void launch_pipe_prepare(const PipeArgs &a, int grid, cudaStream_t s);
void launch_pipe_regroup(const PipeArgs &a, int grid, cudaStream_t s);
void launch_pipe_masks(const PipeArgs &a, int grid, cudaStream_t s);
void launch_pipe_k2sort(const PipeArgs &a, int grid, cudaStream_t s);   // scan + scatter
void launch_pipe_k2(const PipeArgs &a, int grid, cudaStream_t s);
void launch_pipe_one(const PipeArgs &a, int grid, cudaStream_t s);
void launch_pipe_two(const PipeArgs &a, int grid, cudaStream_t s);
void launch_pipe_lift(const PipeArgs &a, int grid, cudaStream_t s);
void launch_pipe_leftover(const PipeArgs &a, cudaStream_t s);
int pipe_ctas_per_sm();

// ---- --write-details text (wfl_details.cu) --------------------------------------------------------
// One (contig, evaluation index) run of the details dump: entries [start, start + len).
struct DetSeg {
    long long start;
    int len, contig, iter, pad;
};

struct DetTextArgs {
    DevBatch b;
    DevTax t;
    DevParams P;
    const int *anc;                // ancestor table (wfl_set_taxonomy): row l = l-th ancestor of every node
    int anc_rows;
    // the dump: contig, evaluation index, clade, raw locus index within the contig, score
    const int32_t *dc, *di, *dc_clade, *dl;
    const double *ds;
    long long n_dump;
    DetSeg *found;                 // segments kernel: every run of the dump, unordered ...
    unsigned int *n_found;         // ... and their number
    const DetSeg *seg;             // rows kernel: segments in row order
    const int *list;               // segments to do: list[0, n_list), or null: [s0, s0 + n_list)
    long long s0, n_list;
    const char *cname;             // contig names by contig index: cname[cname_off[c], cname_off[c + 1])
    const int64_t *cname_off;
    const char *tname;             // clade names by node index
    const int64_t *tname_off;
    char *scratch;                 // `slice` bytes per warp
    long long slice;
    int *defer;                    // segments whose scratch exceeds the slice, their number and the largest need
    unsigned int *n_defer;
    unsigned long long *max_need;
    long long *seg_bytes;          // length pass (text == null): bytes of every segment
    char *text;                    // write pass: the text of the segments, segment si at text_off[si] - text_base
    const long long *text_off;
    long long text_base;
    unsigned int *err;             // scores outside the formatter's exact range
};
void launch_details_segments(const DetTextArgs &a, cudaStream_t s);
void launch_details_rows(const DetTextArgs &a, long long warps, cudaStream_t s);
void launch_format3(const double *x, long long n, char *text, int *len, unsigned int *err, cudaStream_t s);

// ---- the wide scoring batch built from a parser's resident hit columns (wfl_resident_batch.cu) ------------------
struct ResBatchArgs {
    // the parser's columns, one entry per parsed row
    const int32_t *qstart, *qend, *tcode;
    const double *score, *scov;
    const int8_t *strand;
    const unsigned long long *rawmask;
    // the batch: contig c takes rows [hit_src[c], hit_src[c] + hit_off[c + 1] - hit_off[c])
    const int64_t *hit_off, *hit_src;
    long long n, nh;
    const int32_t *slot_node;      // distinct-taxon slot -> node index
    int n_slots, n_nodes;
    const int32_t *sys_perm;       // [64] raw system bit -> bit in the sorted system list; null: no systems, hits sorted
    // outputs: the engine's wide input columns
    int32_t *o_qstart, *o_qend, *o_taxon;
    double *o_score, *o_scov;
    int8_t *o_strand;
    uint32_t *o_sysmask;
    unsigned long long *red;       // [0] hits with an unusable slot, [1] bits of the largest finite score > 0, [2] largest node
    // sort (Batch.sort_hits): quantised (taxon << bits_s | q, row) or lexsort (taxon, -score, row) keys
    bool quantised;
    int bits_s;
    double smax;
    const int *list;               // contigs of the second launch, or null: every contig whose keys fit `slice`
    long long n_list;
    char *scratch;                 // `slice` bytes per warp
    long long slice;
};
void launch_resident_gather(const ResBatchArgs &a, int sm_count, cudaStream_t s);   // checks, reductions; copies if unsorted
void launch_resident_sort(const ResBatchArgs &a, long long warps, cudaStream_t s);

// Compaction (K10): CSR of melded members in contig order + contig indices grouped by call.
struct CompactArgs {
    int64_t n;
    DevOut o;
    int64_t *member_off;      // [n+1]
    int32_t *n_members_a;     // [n]
    int32_t *members;         // compacted
    int64_t members_cap;
    int64_t *call_counts;     // [3]
    int64_t *call_index;      // [n]
    int64_t *scan_tmp;        // [4 * n_blocks] scratch
    int64_t *totals;          // [4]: members, lgt, no_lgt, unclassified
};
int launch_compaction(const CompactArgs &a, cudaStream_t s);   // returns kernels launched
size_t compaction_scratch_elems(int64_t n);

}  // namespace wfl
