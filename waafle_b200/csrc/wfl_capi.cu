// C ABI of the engine (include/waafle_b200.h): handle, device memory, H2D / launch / D2H.
// Plain CUDA runtime -- no torch types anywhere near the boundary.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <string>
#include <vector>

#include "wfl_device.cuh"
#include "wfl_parser.cuh"

using namespace wfl;

namespace {

struct Buf {
    void *p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct wfl_engine {
    int device = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr, copy_stream = nullptr, stream2 = nullptr;
    cudaEvent_t ev_join = nullptr;
    int n_slots = 2;                     // sub-batches alternate between two compute streams
    cudaEvent_t ev[8] = {};
    std::vector<cudaEvent_t> chunk_ev;
    size_t chunk_bytes = size_t(48) << 20;   // H2D chunk size of the pipelined plugin call
    std::string err;
    bool have_params = false, have_tax = false, have_batch = false, have_results = false;
    DevParams P{};
    DevTax tax{};
    DevBatch b{};
    DevOut o{};
    int64_t n = 0, nh = 0, nl = 0;
    int S = 0;
    bool packed = false;                 // the resident batch is in the compact wire format
    // options (wfl_set_option / environment)
    bool exact = false;                  // every contig through the exact pipeline
    int fast_hcap = 0, fast_mcap = 0, fast_tcap = 0, fast_ncap = 0;   // slice capacities of the fast kernel (0 = from the batch)
    double fast_hscale = 1.6;            // first-pass hit capacity as a multiple of the mean hits per contig
    int fast_passes = 2;                 // 1: no second pass with a larger slice
    size_t pipe_pool_bytes = size_t(8192) << 20;
    size_t k2_cap_override = 0;
    bool chunk_fixed = false;
    // device buffers (grow-only)
    Buf tx[4], anc, in[12], out[18], ctr, work, scratch, cm[5], dbg[4], plan_index, plan_data;
    Buf fb_list, fast_scratch, fast_wq, blob, status_tmp;
    Buf rb_src, rb_lut, rb_perm, rb_red, rb_list, rb_scratch;   // wfl_upload_parsed: its inputs, reductions, sort scratch
    Buf det[6];                          // --write-details dump: contig, iteration, clade, locus, score, count
    int64_t det_cap = 0, det_used = 0;
    // --write-details text (wfl_details.cu): clade names of the taxonomy, state of the last wfl_details_prepare
    Buf tname, tname_off, cname, cname_off, dt_found, dt_seg, dt_off, dt_bytes, dt_scratch, dt_defer[2], dt_ctr, dt_text;
    bool have_tnames = false, dt_ready = false;
    std::vector<int64_t> dt_seg_off;     // [segments + 1] byte offset of every segment in the table
    std::vector<int64_t> dt_rank_seg;    // [n_order + 1] first segment of every position of the caller's contig order
    size_t fast_scratch_slot = 0;        // bytes of fast-kernel scratch per compute stream
    bool chunks_pool_bound = false;      // the current chunk plan was cut for the exact pipeline's workspace pool
    int plan_nmax = 0;
    int tax_max_depth = 0, anc_rows = 0;
    FastCfg fcfgp{};                    // pairs pass: first-pass capacities with a large survivor-pair list
    FastCfg fcfg{}, fcfg2{};            // first pass (all contigs) / second pass (capacity overflows, larger slice)
    int fast_grid = 0, fast_grid2 = 0, fast_gridp = 0;
    int64_t cfg_key[4] = {-1, -1, -1, -1};
    // exact pipeline state
    Buf pipe_pool[2], pipe_ctg, pipe_lists[2], pipe_cnt[2], pipe_wq[2], k2_desc[2], k2_order[2], k2_keys[2], k2_meta[2];
    std::vector<int64_t> h_hit_off, h_locus_off;
    std::vector<int64_t> chunks;         // contig boundaries of the sub-batches of the current batch
    bool chunks_streamed = false;        // their H2D copies are in flight on copy_stream (plugin call)
    wfl_stats stats{};
    int64_t members_total = 0;
};

namespace {

// WFL_TRACE=1: host-side timeline of a plugin call on stderr (milliseconds since the call started)
static bool g_trace = getenv("WFL_TRACE") != nullptr;
static std::chrono::steady_clock::time_point g_t0;
static void trace(const char *what) {
    if (!g_trace) return;
    if (!strcmp(what, "begin")) g_t0 = std::chrono::steady_clock::now();
    fprintf(stderr, "[wfl] %8.3f ms  %s\n",
            std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - g_t0).count(), what);
}

bool set_err(wfl_engine *e, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    e->err = buf;
    return false;
}

#define CU(call)                                                                          \
    do {                                                                                  \
        cudaError_t _err = (call);                                                        \
        if (_err != cudaSuccess) {                                                        \
            set_err(e, "%s failed: %s", #call, cudaGetErrorString(_err));                 \
            return WFL_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)

int ensure(wfl_engine *e, Buf &b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return WFL_OK;
    if (b.p) CU(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + bytes / 8;
    CU(cudaMalloc(&b.p, want));
    b.cap = want;
    return WFL_OK;
}

template <class T>
int upload(wfl_engine *e, Buf &b, const T *src, size_t n, const T **dst, cudaStream_t st = nullptr) {
    int rc = ensure(e, b, n * sizeof(T));
    if (rc) return rc;
    if (n) CU(cudaMemcpyAsync(b.p, src, n * sizeof(T), cudaMemcpyHostToDevice, st ? st : e->stream));
    *dst = static_cast<const T *>(b.p);
    return WFL_OK;
}

template <class T>
int outbuf(wfl_engine *e, Buf &b, size_t n, T **dst) {
    int rc = ensure(e, b, n * sizeof(T));
    if (rc) return rc;
    *dst = static_cast<T *>(b.p);
    return WFL_OK;
}


// Host twin of the kernel's build_plan(): numpy's pairwise split tree over n elements, flattened
// (numpy/_core/src/umath/loops_utils.h.src: leaves <= 128, split at n/2 - (n/2) % 8).
void host_build_plan(int n, std::vector<uint16_t> &data, PlanEntry &pe) {
    pe.off = (uint32_t)data.size();
    int sz[64], ch[64], sp = 0, nset = 0;
    uint8_t k8[5] = {0, 0, 0, 0, 0};
    sz[0] = n;
    ch[0] = 0;
    sp = 1;
    uint32_t cnt = 0;
    while (sp > 0) {
        int m = sz[--sp], c = ch[sp];
        if (m <= 128) {
            data.push_back((uint16_t)(m | (c << 8)));
            ++cnt;
            if (m >= 8 && nset <= 4) {
                uint8_t k = (uint8_t)(m >> 3);
                int j = 0;
                while (j < nset && j < 4 && k8[j] < k) ++j;
                if (j == nset || (j < 4 && k8[j] != k)) {
                    if (nset < 4) {
                        for (int q = nset; q > j; --q) k8[q] = k8[q - 1];
                        k8[j] = k;
                    }
                    ++nset;
                }
            }
        } else {
            int n2 = m / 2;
            n2 -= n2 % 8;
            sz[sp] = m - n2;
            ch[sp++] = c + 1;
            sz[sp] = n2;
            ch[sp++] = 0;
        }
    }
    pe.nleaf = cnt;
    if (nset > 4) k8[0] = k8[1] = k8[2] = k8[3] = 0;
    pe.k8 = (uint32_t)k8[0] | ((uint32_t)k8[1] << 8) | ((uint32_t)k8[2] << 16) | ((uint32_t)k8[3] << 24);
}


// Leaf plans for every gene length up to `want` (capped): built once, kept on the device.
int ensure_plan_table(wfl_engine *e, int want) {
    const int cap = 16384;
    want = std::min(std::max(want, 4096), cap);
    if (e->plan_nmax >= want) return WFL_OK;
    std::vector<PlanEntry> index((size_t)want + 1);
    std::vector<uint16_t> data;
    data.reserve((size_t)want * want / 150 + 1024);
    index[0] = PlanEntry{0, 0, 0};
    for (int n = 1; n <= want; ++n) host_build_plan(n, data, index[n]);
    const PlanEntry *di;
    const uint16_t *dd;
    int rc;
    if ((rc = upload(e, e->plan_index, index.data(), index.size(), &di))) return rc;
    if ((rc = upload(e, e->plan_data, data.data(), data.size(), &dd))) return rc;
    CU(cudaStreamSynchronize(e->stream));
    e->plan_nmax = want;
    return WFL_OK;
}

int alloc_outputs(wfl_engine *e) {
    const size_t n = (size_t)e->n, nl = (size_t)e->nl, S = (size_t)e->S;
    int rc = 0;
    DevOut &o = e->o;
    rc |= outbuf(e, e->out[0], n, &o.call);
    rc |= outbuf(e, e->out[1], n, &o.direction);
    rc |= outbuf(e, e->out[2], n, &o.lifts);
    rc |= outbuf(e, e->out[3], n, &o.clade1);
    rc |= outbuf(e, e->out[4], n, &o.clade2);
    rc |= outbuf(e, e->out[5], n, &o.lca);
    rc |= outbuf(e, e->out[6], n, &o.best1);
    rc |= outbuf(e, e->out[7], n, &o.best2);
    rc |= outbuf(e, e->out[8], n, &o.crit);
    rc |= outbuf(e, e->out[9], n, &o.rank);
    rc |= outbuf(e, e->out[10], nl, &o.synteny);
    rc |= outbuf(e, e->out[11], nl, &o.locus_flags);
    rc |= outbuf(e, e->out[12], nl * S, &o.ann_winner);
    rc |= outbuf(e, e->out[13], n, &o.n_mem_a);
    rc |= outbuf(e, e->out[14], n, &o.n_mem_b);
    rc |= outbuf(e, e->out[15], n, &o.mem_pos);
    rc |= outbuf(e, e->out[17], n, &o.status);
    if (rc) return WFL_ERR_CUDA;
    size_t pool = std::max<size_t>(e->out[16].cap / sizeof(int32_t), std::max<size_t>(2 * n, 1 << 16));
    rc = outbuf(e, e->out[16], pool, &o.mem_pool);
    o.mem_pool_cap = (int64_t)(e->out[16].cap / sizeof(int32_t));
    return rc;
}

// One host-side description of a batch in either wire format.
struct HostBatch {
    int64_t n = 0, nh = 0, nl = 0;
    const int64_t *hit_off = nullptr, *locus_off = nullptr;
    const int32_t *locus_start = nullptr, *locus_end = nullptr;
    const int8_t *locus_strand = nullptr;
    bool packed = false;
    // hit columns: (source pointer, element size); wide: qstart qend taxon score scov strand sysmask,
    // packed: qstart16 qend16 tax16 score sysmask8
    const void *col[7] = {};
    int esz[7] = {};
    int ncol = 0;
};

HostBatch host_batch(const wfl_batch *in, int S) {
    HostBatch h;
    h.n = in->n_contigs; h.nh = in->n_hits; h.nl = in->n_loci;
    h.hit_off = in->hit_off; h.locus_off = in->locus_off;
    h.locus_start = in->locus_start; h.locus_end = in->locus_end; h.locus_strand = in->locus_strand;
    const void *c[7] = {in->hit_qstart, in->hit_qend, in->hit_taxon, in->hit_score, in->hit_scov, in->hit_strand,
                        S > 0 ? in->hit_sysmask : nullptr};
    const int z[7] = {4, 4, 4, 8, 8, 1, 4};
    for (int i = 0; i < 7; ++i) { h.col[i] = c[i]; h.esz[i] = z[i]; }
    h.ncol = 7;
    return h;
}

HostBatch host_batch(const wfl_packed_batch *in, int S) {
    HostBatch h;
    h.packed = true;
    h.n = in->n_contigs; h.nh = in->n_hits; h.nl = in->n_loci;
    h.hit_off = in->hit_off; h.locus_off = in->locus_off;
    h.locus_start = in->locus_start; h.locus_end = in->locus_end; h.locus_strand = in->locus_strand;
    const void *c[5] = {in->hit_qstart16, in->hit_qend16, in->hit_tax16, in->hit_score, S > 0 ? in->hit_sysmask8 : nullptr};
    const int z[5] = {2, 2, 2, 8, 1};
    for (int i = 0; i < 5; ++i) { h.col[i] = c[i]; h.esz[i] = z[i]; }
    h.ncol = 5;
    return h;
}

size_t hit_row_bytes(const HostBatch &h) {
    size_t r = 0;
    for (int i = 0; i < h.ncol; ++i) r += h.col[i] ? (size_t)h.esz[i] : 0;
    return r;
}

int check_host_batch(wfl_engine *e, const HostBatch &h) {
    if (h.n < 0 || h.nh < 0 || h.nl < 0) { set_err(e, "bad batch sizes"); return WFL_ERR_ARG; }
    if (h.nh >= (1ll << 31) || h.nl >= (1ll << 31) || h.n >= (1ll << 31)) {
        set_err(e, "batch too large: contigs, hits and loci must each be < 2^31 per batch");
        return WFL_ERR_ARG;
    }
    bool null_hit = false;
    for (int i = 0; i < h.ncol; ++i) {
        const bool optional = i == h.ncol - 1;   // the sysmask column
        if (h.nh && !h.col[i] && !optional) null_hit = true;
    }
    if (!h.hit_off || !h.locus_off || null_hit || (h.nl && (!h.locus_start || !h.locus_end || !h.locus_strand))) {
        set_err(e, "null array in batch");
        return WFL_ERR_ARG;
    }
    if (e->P.p.n_systems > 0 && h.nh && !h.col[h.ncol - 1]) {
        set_err(e, "n_systems > 0 but hit_sysmask is null");
        return WFL_ERR_ARG;
    }
    if (h.packed && (e->tax.n_nodes > WFL_PACKED_MAX_NODES || e->P.p.n_systems > WFL_PACKED_MAX_SYSTEMS)) {
        set_err(e, "compact wire format needs <= %d taxonomy nodes and <= %d annotation systems", WFL_PACKED_MAX_NODES,
                WFL_PACKED_MAX_SYSTEMS);
        return WFL_ERR_ARG;
    }
    if (h.hit_off[0] != 0 || h.locus_off[0] != 0 || h.hit_off[h.n] != h.nh || h.locus_off[h.n] != h.nl) {
        set_err(e, "CSR offsets do not span the hit / locus arrays");
        return WFL_ERR_ARG;
    }
    for (int64_t c = 0; c < h.n; ++c)
        if (h.hit_off[c + 1] < h.hit_off[c] || h.locus_off[c + 1] < h.locus_off[c]) {
            set_err(e, "CSR offsets are not monotone at contig %lld", (long long)c);
            return WFL_ERR_ARG;
        }
    return WFL_OK;
}

// device pointer of hit column i of the resident batch
void *&dev_col(wfl_engine *e, int i) { return e->in[2 + i].p; }

void bind_device_batch(wfl_engine *e) {
    DevBatch &b = e->b;
    b.hit_qstart = b.hit_qend = b.hit_taxon = nullptr;
    b.hit_score = b.hit_scov = nullptr;
    b.hit_strand = nullptr;
    b.hit_sysmask = nullptr;
    b.hit_qstart16 = b.hit_qend16 = b.hit_tax16 = nullptr;
    b.hit_sysmask8 = nullptr;
    if (e->packed) {
        b.hit_qstart16 = static_cast<const uint16_t *>(dev_col(e, 0));
        b.hit_qend16 = static_cast<const uint16_t *>(dev_col(e, 1));
        b.hit_tax16 = static_cast<const uint16_t *>(dev_col(e, 2));
        b.hit_score = static_cast<const double *>(dev_col(e, 3));
        if (e->S > 0) b.hit_sysmask8 = static_cast<const uint8_t *>(dev_col(e, 4));
    } else {
        b.hit_qstart = static_cast<const int32_t *>(dev_col(e, 0));
        b.hit_qend = static_cast<const int32_t *>(dev_col(e, 1));
        b.hit_taxon = static_cast<const int32_t *>(dev_col(e, 2));
        b.hit_score = static_cast<const double *>(dev_col(e, 3));
        b.hit_scov = static_cast<const double *>(dev_col(e, 4));
        b.hit_strand = static_cast<const int8_t *>(dev_col(e, 5));
        if (e->S > 0) b.hit_sysmask = static_cast<const uint32_t *>(dev_col(e, 6));
    }
    b.locus_start = static_cast<const int32_t *>(e->in[9].p);
    b.locus_end = static_cast<const int32_t *>(e->in[10].p);
    b.locus_strand = static_cast<const int8_t *>(e->in[11].p);
}

// Cut the batch into sub-batches of whole contigs.
//  * exact pipeline: a sub-batch's intermediate state must fit the workspace pool;
//  * plugin call (streaming): a sub-batch is also the unit that crosses PCIe on the copy stream while its
//    predecessor is scored: a small first chunk (the kernels start early), then equal chunks, at most ~12 per call
//    (every chunk costs a launch chain that ends on its slowest contig).
bool uses_fast_path(const wfl_engine *e) {
    return !e->exact && e->det_cap == 0 && e->P.p.min_overlap > 0.0 && e->nl <= 32 * e->n;
}

void plan_chunks(wfl_engine *e, const int64_t *hoff, const int64_t *loff, bool streaming, size_t hit_row) {
    e->chunks.clear();
    e->chunks.push_back(0);
    const int64_t n = e->n;
    if (n <= 0) return;
    const bool pool_bound = !uses_fast_path(e);   // the exact pipeline's sub-batches must fit its workspace pool
    e->chunks_pool_bound = pool_bound;
    std::vector<size_t> target;
    if (streaming) {
        const size_t total = (size_t)hoff[n] * hit_row;
        // fast path: one launch per chunk, ~12 chunks hide the kernels under the transfer; exact pipeline (long contigs,
        // --exact-scores): every chunk costs a 9-launches-per-level chain that needs thousands of contigs to fill the GPU
        // (measured at BASELINE configs[3]: 4 000 contigs in 12 chunks 136 ms per call, in one chunk 43 ms)
        const size_t per_contig = total / (size_t)n + 1;
        const size_t full = e->chunk_fixed ? e->chunk_bytes
                                           : std::max(e->chunk_bytes, pool_bound ? std::max(total / 3 + 1, 8192 * per_contig)
                                                                                 : total / 12 + 1);
        const size_t first = std::min(full / 4, e->chunk_bytes);
        size_t rem = total;
        target.push_back(std::min(rem, first));
        rem -= target.back();
        if (rem % full) { target.push_back(rem % full); rem -= rem % full; }   // the odd piece goes early
        for (; rem > 0; rem -= full) target.push_back(full);
    }
    int64_t c0 = 0;
    size_t k = 0;
    while (c0 < n) {
        int64_t c1 = c0;
        size_t est = 0;
        const size_t goal = k < target.size() ? target[k] : (target.empty() ? ~size_t(0) : target.back());
        for (;;) {
            // workspace estimate per contig (records + table + level arrays), see wfl_pipeline.cu
            const size_t h = (size_t)(hoff[c1 + 1] - hoff[c1]), g = (size_t)(loff[c1 + 1] - loff[c1]);
            est += 190 * h + 96 * g + 9000;
            ++c1;
            if (c1 >= n) break;
            if (streaming && (size_t)(hoff[c1 + 1] - hoff[c0]) * hit_row > goal) break;
            if (pool_bound && est + 190 * (size_t)(hoff[c1 + 1] - hoff[c1]) + 9000 > e->pipe_pool_bytes) break;
        }
        e->chunks.push_back(c1);
        c0 = c1;
        ++k;
    }
}

// All H2D copies of the plugin call, chunk by chunk on the copy stream, one event per chunk.
int issue_chunk_copies(wfl_engine *e, const HostBatch &src) {
    const int64_t *hoff = src.hit_off, *loff = src.locus_off;
    cudaStream_t cs = e->copy_stream;
    for (size_t k = 0; k + 1 < e->chunks.size(); ++k) {
        const int64_t c0 = e->chunks[k], c1 = e->chunks[k + 1];
        const size_t h0 = (size_t)hoff[c0], h1 = (size_t)hoff[c1];
        const size_t l0 = (size_t)loff[c0], l1 = (size_t)loff[c1];
        for (int i = 0; i < src.ncol; ++i)
            if (src.col[i] && h1 > h0)
                CU(cudaMemcpyAsync(static_cast<char *>(dev_col(e, i)) + h0 * src.esz[i],
                                   static_cast<const char *>(src.col[i]) + h0 * src.esz[i], (h1 - h0) * src.esz[i],
                                   cudaMemcpyHostToDevice, cs));
        if (l1 > l0) {
            CU(cudaMemcpyAsync(static_cast<int32_t *>(e->in[9].p) + l0, src.locus_start + l0, (l1 - l0) * 4, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(static_cast<int32_t *>(e->in[10].p) + l0, src.locus_end + l0, (l1 - l0) * 4, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(static_cast<int8_t *>(e->in[11].p) + l0, src.locus_strand + l0, (l1 - l0), cudaMemcpyHostToDevice, cs));
        }
        if (e->chunk_ev.size() <= k) {
            cudaEvent_t evn;
            CU(cudaEventCreateWithFlags(&evn, cudaEventDisableTiming));
            e->chunk_ev.push_back(evn);
        }
        CU(cudaEventRecord(e->chunk_ev[k], cs));
    }
    CU(cudaEventRecord(e->ev[5], cs));   // end of the last H2D chunk
    e->chunks_streamed = true;
    return WFL_OK;
}

// One sub-batch through the exact multi-kernel pipeline (wfl_pipeline.cu): the contig range [c0, c0 + n_work) or, with
// `list`, the n_work contigs it names.  `hits` bounds the K2 group list; `grow` scales the capacities of a replay.
int launch_pipeline(wfl_engine *e, DevCounters *ctr, const int *list, int64_t c0, int64_t n_work, size_t hits, int slot,
                    size_t grow, long long dbg_contig = -1) {
    cudaStream_t stream = slot ? e->stream2 : e->stream;
    const int L = std::min(std::max(e->tax_max_depth + 1 - e->P.p.jump_taxonomy, 1), 64);
    int rc;
    char *pool;
    PipeCtg *ctg;
    int *lists, *cnt;
    unsigned long long *wq;
    const size_t n = (size_t)e->n;
    const size_t pool_want = grow > 1 ? std::min<size_t>(std::max<size_t>(e->pipe_pool_bytes, size_t(64) << 20) * grow, size_t(64) << 30)
                                      : std::min<size_t>(e->pipe_pool_bytes, 200 * (size_t)e->nh + 9200 * n + 96 * (size_t)e->nl + (size_t(64) << 20));
    if ((rc = outbuf(e, e->pipe_pool[slot], std::max<size_t>(pool_want, e->pipe_pool[slot].cap), &pool))) return rc;
    if ((rc = outbuf(e, e->pipe_ctg, n, &ctg))) return rc;
    if ((rc = outbuf(e, e->pipe_lists[slot], 4 * n + 16, &lists))) return rc;
    if ((rc = outbuf(e, e->pipe_cnt[slot], 3 * 66 + 8, &cnt))) return rc;
    if ((rc = outbuf(e, e->pipe_wq[slot], 6 * 66 + 8, &wq))) return rc;
    CU(cudaMemsetAsync(cnt, 0, (3 * 66 + 8) * sizeof(int), stream));
    CU(cudaMemsetAsync(wq, 0, (6 * 66 + 8) * sizeof(unsigned long long), stream));
    PipeArgs pa{};
    pa.b = e->b; pa.t = e->tax; pa.o = e->o; pa.P = e->P; pa.ctr = ctr;
    pa.pool = pool; pa.pool_used = wq; pa.pool_cap = std::min<size_t>(e->pipe_pool[slot].cap, std::max<size_t>(pool_want, 16));
    pa.ctg = ctg;
    pa.plan_nmax = e->plan_nmax;
    pa.plan_index = static_cast<const PlanEntry *>(e->plan_index.p);
    pa.plan_data = static_cast<const uint16_t *>(e->plan_data.p);
    K2Meta *k2meta = nullptr;
    {
        const size_t cap = (e->k2_cap_override && grow <= 1) ? e->k2_cap_override : (hits * 5 / 4 + 4096) * grow;
        if ((rc = outbuf(e, e->k2_desc[slot], cap, &pa.k2_desc))) return rc;
        if ((rc = outbuf(e, e->k2_order[slot], cap, &pa.k2_order))) return rc;
        if ((rc = outbuf(e, e->k2_keys[slot], cap, &pa.k2_keys))) return rc;
        if ((rc = outbuf(e, e->k2_meta[slot], 66, &k2meta))) return rc;
        pa.k2_cap = cap;
        CU(cudaMemsetAsync(k2meta, 0, 66 * sizeof(K2Meta), stream));
    }
    if (e->det_cap > 0) {
        pa.det_count = static_cast<unsigned long long *>(e->det[5].p);
        pa.det_cap = e->det_cap;
        pa.det_contig = static_cast<int32_t *>(e->det[0].p);
        pa.det_iter = static_cast<int32_t *>(e->det[1].p);
        pa.det_clade = static_cast<int32_t *>(e->det[2].p);
        pa.det_locus = static_cast<int32_t *>(e->det[3].p);
        pa.det_score = static_cast<double *>(e->det[4].p);
    }
    pa.dbg_contig = dbg_contig;
    if (dbg_contig >= 0) {
        pa.dbg_clade = static_cast<int32_t *>(e->dbg[0].p);
        pa.dbg_locus = static_cast<int32_t *>(e->dbg[1].p);
        pa.dbg_score = static_cast<double *>(e->dbg[2].p);
        pa.dbg_cap = (long long)(e->dbg[0].cap / sizeof(int32_t));
        pa.dbg_count = static_cast<long long *>(e->dbg[3].p);
    }
    int *lst[4] = {lists, lists + n, lists + 2 * n, lists + 3 * n};
    int *cnt_act = cnt, *cnt_two = cnt + 66, *cnt_lift = cnt + 2 * 66;
    const int grid = e->sm_count * pipe_ctas_per_sm();
    pa.wq = wq + 1;
    pa.work_base = c0; pa.n_work = n_work; pa.work_list = list;
    pa.list_act = lst[0]; pa.cnt_act = &cnt_act[0];
    launch_pipe_prepare(pa, (int)std::max<int64_t>(1, std::min<int64_t>(grid, n_work)), stream);
    for (int lvl = 0; lvl < L; ++lvl) {
        pa.list_act = lst[lvl & 1]; pa.cnt_act = &cnt_act[lvl];
        pa.list_next = lst[(lvl + 1) & 1]; pa.cnt_next = &cnt_act[lvl + 1];
        pa.list_two = lst[2]; pa.cnt_two = &cnt_two[lvl];
        pa.list_lift = lst[3]; pa.cnt_lift = &cnt_lift[lvl];
        pa.k2_meta = k2meta + lvl;
        pa.wq = wq + 2 + 6 * lvl;
        launch_pipe_regroup(pa, grid, stream);
        pa.wq = wq + 3 + 6 * lvl;
        launch_pipe_k2sort(pa, grid, stream);
        launch_pipe_k2(pa, grid, stream);
        pa.wq = wq + 4 + 6 * lvl;
        launch_pipe_masks(pa, grid, stream);
        pa.wq = wq + 5 + 6 * lvl;
        launch_pipe_one(pa, grid, stream);
        pa.wq = wq + 6 + 6 * lvl;
        launch_pipe_two(pa, grid, stream);
        pa.wq = wq + 7 + 6 * lvl;
        launch_pipe_lift(pa, grid, stream);
    }
    pa.list_act = lst[L & 1]; pa.cnt_act = &cnt_act[L];
    launch_pipe_leftover(pa, stream);
    CU(cudaGetLastError());
    e->stats.kernel_launches += 2 + 9 * L;
    return WFL_OK;
}

// The exact pipeline over an explicit contig list (fast-path fallbacks, workspace replays), cut into sub-batches whose
// estimated workspace fits the pool.
int run_pipeline_list(wfl_engine *e, DevCounters *ctr, const std::vector<int> &list, size_t grow) {
    if (list.empty()) return WFL_OK;
    int rc;
    int *dl;
    if ((rc = outbuf(e, e->work, list.size(), &dl))) return rc;
    CU(cudaMemcpyAsync(dl, list.data(), list.size() * sizeof(int), cudaMemcpyHostToDevice, e->stream));
    const size_t pool = grow > 1 ? std::min<size_t>(std::max<size_t>(e->pipe_pool_bytes, size_t(64) << 20) * grow, size_t(64) << 30)
                                 : e->pipe_pool_bytes;
    size_t i0 = 0;
    while (i0 < list.size()) {
        size_t i1 = i0, est = 0, hits = 0;
        while (i1 < list.size()) {
            const int c = list[i1];
            const size_t h = (size_t)(e->h_hit_off[c + 1] - e->h_hit_off[c]), g = (size_t)(e->h_locus_off[c + 1] - e->h_locus_off[c]);
            const size_t need = 190 * h + 96 * g + 9000;
            if (i1 > i0 && est + need > pool) break;
            est += need;
            hits += h;
            ++i1;
        }
        if ((rc = launch_pipeline(e, ctr, dl + i0, 0, (int64_t)(i1 - i0), hits, 0, grow))) return rc;
        i0 = i1;
    }
    return WFL_OK;
}

// Capacities of the fast kernel's shared-memory slices, chosen from the shape of the batch (options override).
// First pass: sized for the bulk of the contigs (hits per contig up to ~1.6x the mean), so that as many warps as possible
// are resident; second pass: the contigs that overflowed, with a slice ~3x as large.
static void fit_layout(wfl_engine *e, FastCfg &F, int H, int M, int T, int N, int Sc) {
    for (;;) {
        fast_layout(F, H, M, T, N, Sc, e->P.p.n_systems);
        if ((size_t)fast_warps_per_cta() * F.slice_bytes + 1024 <= e->smem_optin) break;
        // does not fit one CTA: shrink the largest consumers
        if (N > 96) N = std::max(96, N * 3 / 4);
        if (T > 64) T = std::max(64, T * 3 / 4);
        if (M > 128) M = std::max(128, M * 3 / 4);
        if (H > 128) H = std::max(128, H * 3 / 4);
        if (Sc > 64) Sc = std::max(64, Sc / 2);
        if (N <= 96 && T <= 64 && M <= 128 && H <= 128) break;
    }
}

void choose_fast_cfg(wfl_engine *e) {
    int64_t hmax = 0;
    for (int64_t c = 0; c < e->n; ++c) hmax = std::max(hmax, e->h_hit_off[c + 1] - e->h_hit_off[c]);
    const int64_t key[4] = {e->nh, e->nl, e->n * 2 + (e->packed ? 1 : 0), hmax * 64 + e->P.p.n_systems};
    if (!memcmp(key, e->cfg_key, sizeof key)) return;
    const double hbar = e->n > 0 ? (double)e->nh / (double)e->n : 0.0;        // hits per contig
    auto r16 = [](double x) { return (int)((x + 15.0) / 16.0) * 16; };
    const double hq = std::min((double)hmax, e->fast_hscale * hbar);
    const int H = e->fast_hcap ? e->fast_hcap : std::min(16384, std::max(64, r16(hq + 16)));
    const int M = e->fast_mcap ? e->fast_mcap : H;   // entries (hit x locus matches) ~ hits: a few hits match two loci, ~5 % none
    const int T = e->fast_tcap ? e->fast_tcap : std::min(4096, std::max(64, r16(0.42 * H + 16)));
    const int N = e->fast_ncap ? e->fast_ncap : std::min(16384, std::max(96, r16(0.6 * H + 32)));
    fit_layout(e, e->fcfg, H, M, T, N, 64);
    fit_layout(e, e->fcfgp, H, M, T, N, 1024);          // same slice, room for many two-clade survivor pairs
    fit_layout(e, e->fcfg2, 3 * H, 3 * M, 3 * T, 3 * N, 2048);
    e->fast_grid = e->sm_count * std::max(1, fast_ctas_per_sm(e->fcfg, e->packed, 0));
    e->fast_grid2 = e->sm_count * std::max(1, fast_ctas_per_sm(e->fcfg2, e->packed, 0));
    e->fast_gridp = e->sm_count * std::max(1, fast_ctas_per_sm(e->fcfgp, e->packed, 0));
    memcpy(e->cfg_key, key, sizeof key);
}

// One launch of the fused fast-path kernel: pass 0 over the contig range [c0, c0 + n_work), pass 1 over the first
// pass's capacity overflows (list and count on the device).
int launch_fast_pass(wfl_engine *e, DevCounters *ctr, int pass, int64_t c0, int64_t n_work, int launch_idx, int slot) {
    cudaStream_t stream = slot ? e->stream2 : e->stream;
    FastArgs a{};
    a.b = e->b; a.t = e->tax; a.o = e->o; a.P = e->P; a.ctr = ctr;
    // pass 0: every contig; pass 1 ("pairs"): first-pass contigs whose survivor-pair list overflowed, same slice with a large
    // Scap; pass 2: every other capacity overflow of passes 0 / 1, slice ~3x as large; what that cannot hold: exact pipeline
    a.cfg = pass == 0 ? e->fcfg : pass == 1 ? e->fcfgp : e->fcfg2;
    a.wq = static_cast<unsigned long long *>(e->fast_wq.p) + launch_idx;
    int *fb_a = static_cast<int *>(e->fb_list.p), *fb_b = fb_a + e->n + 1, *fb_p = fb_b + e->n + 1;
    a.fb_final = fb_b;
    a.fb_final_count = &ctr->n_fallback2;
    const bool multi = e->fast_passes > 1;
    if (pass == 0) {
        a.n_work = n_work; a.work_base = c0; a.work_list = nullptr; a.n_work_dev = nullptr;
        a.fb_list = multi ? fb_a : fb_b;
        a.fb_count = multi ? &ctr->n_fallback : &ctr->n_fallback2;
        a.fb_pairs = multi ? fb_p : nullptr;
        a.fb_pairs_count = &ctr->n_fallback_pairs;
    } else if (pass == 1) {
        a.n_work = 0; a.work_base = 0; a.work_list = fb_p; a.n_work_dev = &ctr->n_fallback_pairs;
        a.fb_list = fb_a;
        a.fb_count = &ctr->n_fallback;
    } else {
        a.n_work = 0; a.work_base = 0; a.work_list = fb_a; a.n_work_dev = &ctr->n_fallback;
        a.fb_list = fb_b;
        a.fb_count = &ctr->n_fallback2;
    }
    a.anc = static_cast<const int *>(e->anc.p);
    a.anc_rows = e->anc_rows;
    a.guard = 1e-12;
    {
        int cb = 1;
        while ((1ll << cb) < (long long)e->tax.n_nodes) ++cb;
        a.qbits = std::min(32, 48 - cb);
    }
    a.plan_nmax = e->plan_nmax;
    a.plan_index = static_cast<const PlanEntry *>(e->plan_index.p);
    a.plan_data = static_cast<const uint16_t *>(e->plan_data.p);
    a.scratch = static_cast<char *>(e->fast_scratch.p) + (size_t)slot * e->fast_scratch_slot;   // launches on the two streams overlap
    const int wpc = fast_warps_per_cta();
    const int grid = pass == 2 ? e->fast_grid2 : pass == 1 ? e->fast_gridp : (int)std::max<int64_t>(1, std::min<int64_t>(e->fast_grid, (n_work + wpc - 1) / wpc));
    cudaError_t err = launch_fast(a, e->packed, grid, stream);
    if (err != cudaSuccess) { set_err(e, "fast kernel launch failed: %s", cudaGetErrorString(err)); return WFL_ERR_CUDA; }
    e->stats.kernel_launches++;
    return WFL_OK;
}

template <class T>
int d2h(wfl_engine *e, T *dst, const T *src, size_t n) {
    if (!dst || n == 0) return WFL_OK;
    CU(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, e->stream));
    return WFL_OK;
}

// Queue the D2H copies of every result array; `members` copies that many member entries.
int queue_downloads(wfl_engine *e, wfl_results *out, size_t members) {
    const size_t n = (size_t)e->n, nl = (size_t)e->nl, S = (size_t)e->S;
    const DevOut &o = e->o;
    int rc = 0;
    rc |= d2h(e, out->call, o.call, n);
    rc |= d2h(e, out->direction, o.direction, n);
    rc |= d2h(e, out->lifts, o.lifts, n);
    rc |= d2h(e, out->clade1, o.clade1, n);
    rc |= d2h(e, out->clade2, o.clade2, n);
    rc |= d2h(e, out->lca, o.lca, n);
    rc |= d2h(e, out->best1, o.best1, n);
    rc |= d2h(e, out->best2, o.best2, n);
    rc |= d2h(e, out->crit, o.crit, n);
    rc |= d2h(e, out->rank, o.rank, n);
    rc |= d2h(e, out->synteny, o.synteny, nl);
    rc |= d2h(e, out->locus_flags, o.locus_flags, nl);
    rc |= d2h(e, out->ann_winner, o.ann_winner, nl * S);
    rc |= d2h(e, out->member_off, static_cast<const int64_t *>(e->cm[0].p), n + 1);
    rc |= d2h(e, out->n_members_a, static_cast<const int32_t *>(e->cm[1].p), n);
    rc |= d2h(e, out->members, static_cast<const int32_t *>(e->cm[4].p), members);
    rc |= d2h(e, out->call_counts, static_cast<const int64_t *>(e->cm[2].p), 3);
    rc |= d2h(e, out->call_index, static_cast<const int64_t *>(e->cm[3].p), n);
    return rc ? WFL_ERR_CUDA : WFL_OK;
}

int sync_stream(wfl_engine *e) {
    CU(cudaStreamSynchronize(e->stream));
    e->stats.host_syncs++;
    return WFL_OK;
}

// Score the resident (or in-flight: `streamed`) batch.  Common case = ONE host synchronisation: the fast kernels, the
// compaction and -- with `out` -- the result copies are queued back to back, the counters ride the same stream, and only
// if the fast path handed contigs back (or a workspace overflowed) does the host queue the exact pipeline and a second
// round of compaction + copies.
int run_once(wfl_engine *e, bool streamed, wfl_results *out, bool *restart) {
    *restart = false;
    int rc = alloc_outputs(e);
    if (rc) return rc;
    DevCounters *ctr;
    if ((rc = outbuf(e, e->ctr, 1, &ctr))) return rc;
    int64_t *cm_off, *cm_counts, *cm_index, *cm_totals, *scan_tmp;
    int32_t *cm_na, *cm_members;
    if ((rc = outbuf(e, e->cm[0], (size_t)e->n + 1, &cm_off))) return rc;
    if ((rc = outbuf(e, e->cm[1], (size_t)e->n, &cm_na))) return rc;
    if ((rc = outbuf(e, e->cm[2], 8, &cm_counts))) return rc;
    if ((rc = outbuf(e, e->cm[3], (size_t)e->n, &cm_index))) return rc;
    if ((rc = outbuf(e, e->cm[4], (size_t)e->o.mem_pool_cap, &cm_members))) return rc;
    cm_totals = cm_counts + 4;
    if ((rc = outbuf(e, e->scratch, compaction_scratch_elems(e->n), &scan_tmp))) return rc;
    // the fused fast path holds contigs with <= 32 retained loci; a batch of long contigs (BASELINE configs[3]: 100+ genes)
    // goes straight to the exact pipeline instead of bouncing every contig off the fast kernel first
    const bool use_fast = uses_fast_path(e);
    int *fb_list = nullptr;
    unsigned long long *fwq = nullptr;
    if (use_fast) {
        choose_fast_cfg(e);
        char *fs;
        if ((rc = outbuf(e, e->fb_list, 3 * ((size_t)e->n + 1), &fb_list))) return rc;
        if ((rc = outbuf(e, e->fast_wq, 256, &fwq))) return rc;
        e->fast_scratch_slot = (std::max(std::max((size_t)e->fast_grid * e->fcfg.scratch_bytes, (size_t)e->fast_gridp * e->fcfgp.scratch_bytes), (size_t)e->fast_grid2 * e->fcfg2.scratch_bytes) * fast_warps_per_cta() + 255) & ~(size_t)255;
        if ((rc = outbuf(e, e->fast_scratch, 2 * e->fast_scratch_slot, &fs))) return rc;
        CU(cudaMemsetAsync(fwq, 0, 256 * sizeof(unsigned long long), e->stream));
    }
    CU(cudaMemsetAsync(ctr, 0, sizeof(DevCounters), e->stream));
    if (e->det_cap > 0) {   // --write-details dump (exact pipeline only)
        int32_t *p4;
        double *p8;
        unsigned long long *pc;
        for (int q = 0; q < 4; ++q)
            if ((rc = outbuf(e, e->det[q], (size_t)e->det_cap, &p4))) return rc;
        if ((rc = outbuf(e, e->det[4], (size_t)e->det_cap, &p8)) || (rc = outbuf(e, e->det[5], 1, &pc))) return rc;
        CU(cudaMemsetAsync(pc, 0, sizeof(unsigned long long), e->stream));
    }
    CU(cudaEventRecord(e->ev[1], e->stream));

    if (e->n > 0) {
        if (e->chunks.size() < 2 || e->chunks.back() != e->n || (!e->chunks_streamed && e->chunks_pool_bound != !uses_fast_path(e)))
            plan_chunks(e, e->h_hit_off.data(), e->h_locus_off.data(), false, 29);
        bool used_slot1 = false;
        for (size_t k = 0; k + 1 < e->chunks.size(); ++k) {
            const int64_t c0 = e->chunks[k], c1 = e->chunks[k + 1];
            // sub-batches alternate between two compute streams, so that the tail of one sub-batch's kernels (each ends
            // on its slowest contig) is filled by the next sub-batch's kernels instead of idling the SMs
            const int slot = (e->n_slots > 1 && e->chunks.size() > 2) ? (int)(k & 1) : 0;
            if (slot && !used_slot1) {
                CU(cudaEventRecord(e->ev_join, e->stream));   // orders stream2 after the resets above
                CU(cudaStreamWaitEvent(e->stream2, e->ev_join, 0));
                used_slot1 = true;
            }
            cudaStream_t st = slot ? e->stream2 : e->stream;
            if (streamed && e->chunks_streamed) CU(cudaStreamWaitEvent(st, e->chunk_ev[k], 0));
            if (use_fast) {
                if (k >= 250) { set_err(e, "too many chunks"); return WFL_ERR_ARG; }
                if ((rc = launch_fast_pass(e, ctr, 0, c0, c1 - c0, (int)k, slot))) return rc;
            } else {
                if ((rc = launch_pipeline(e, ctr, nullptr, c0, c1 - c0, (size_t)(e->h_hit_off[c1] - e->h_hit_off[c0]), slot, 1))) return rc;
            }
        }
        if (used_slot1) {
            CU(cudaEventRecord(e->ev_join, e->stream2));
            CU(cudaStreamWaitEvent(e->stream, e->ev_join, 0));
        }
        // second pass: the contigs that overflowed a capacity of the first pass's slice, with a larger slice (their list
        // and count are on the device: no host round trip)
        if (use_fast && e->fast_passes > 1 && ((rc = launch_fast_pass(e, ctr, 1, 0, 0, 254, 0)) || (rc = launch_fast_pass(e, ctr, 2, 0, 0, 255, 0)))) return rc;
    }
    CU(cudaEventRecord(e->ev[2], e->stream));
    trace("kernels launched");

    CompactArgs ca{};
    ca.n = e->n;
    ca.o = e->o;
    ca.member_off = cm_off;
    ca.n_members_a = cm_na;
    ca.call_counts = cm_counts;
    ca.call_index = cm_index;
    ca.scan_tmp = scan_tmp;
    ca.totals = cm_totals;
    ca.members = cm_members;
    ca.members_cap = e->o.mem_pool_cap;

    DevCounters hc{};
    int64_t totals[4] = {0, 0, 0, 0};
    size_t grow = 1;
    for (int attempt = 0;; ++attempt) {
        // (speculative on attempt 0) compaction + counters + result copies, then the one synchronisation
        e->stats.kernel_launches += launch_compaction(ca, e->stream);
        CU(cudaGetLastError());
        CU(cudaEventRecord(e->ev[3], e->stream));
        CU(cudaMemcpyAsync(&hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, e->stream));
        CU(cudaMemcpyAsync(totals, cm_totals, sizeof totals, cudaMemcpyDeviceToHost, e->stream));
        size_t spec_members = 0;
        if (out) {
            CU(cudaEventRecord(e->ev[4], e->stream));
            spec_members = out->members ? (size_t)std::min<int64_t>(out->members_capacity, e->o.mem_pool_cap) : 0;
            if ((rc = queue_downloads(e, out, spec_members))) return rc;
            CU(cudaEventRecord(e->ev[6], e->stream));
        }
        if ((rc = sync_stream(e))) return rc;
        trace("synchronised");
        if (hc.n_badinput) {
            set_err(e, "%llu contig(s) carry a hit taxon index outside the taxonomy", hc.n_badinput);
            return WFL_ERR_ARG;
        }
        if (hc.n_runaway) {
            set_err(e, "Runaway taxonomic recursion in %llu contig(s)", hc.n_runaway);
            return WFL_ERR_RUNAWAY;
        }
        if ((int64_t)hc.mem_pool_used > e->o.mem_pool_cap) {
            // melded-member staging pool too small: grow it and redo the whole batch
            Buf nb;
            if ((rc = ensure(e, nb, (size_t)hc.mem_pool_used * sizeof(int32_t) * 2))) return rc;
            cudaFree(e->out[16].p);
            e->out[16] = nb;
            e->stats.workspace_retries++;
            *restart = true;
            return WFL_OK;
        }
        // contigs for the exact pipeline: fast-path fallbacks (first round) and workspace overflows (status 1)
        std::vector<int> list;
        if (attempt == 0 && use_fast) {
            e->stats.second_pass_contigs = e->fast_passes > 1 ? (int64_t)(hc.n_fallback + hc.n_fallback_pairs) : 0;
            for (int q = 0; q < 8; ++q) e->stats.fallback_reasons[q] = (int64_t)hc.fb_reason[q];
        }
        if (attempt == 0 && hc.n_fallback2) {
            list.resize((size_t)hc.n_fallback2);
            CU(cudaMemcpy(list.data(), fb_list + e->n + 1, list.size() * sizeof(int), cudaMemcpyDeviceToHost));
            std::sort(list.begin(), list.end());
            e->stats.fallback_contigs = (int64_t)list.size();
        } else if (hc.n_overflow) {
            std::vector<uint8_t> st((size_t)e->n);
            CU(cudaMemcpy(st.data(), e->o.status, (size_t)e->n, cudaMemcpyDeviceToHost));
            for (int64_t c = 0; c < e->n; ++c)
                if (st[c] == 1) list.push_back((int)c);
            e->stats.workspace_retries += (int64_t)list.size();
            grow *= 4;
        }
        if (list.empty()) break;
        if (attempt > 8) { set_err(e, "workspace keeps overflowing"); return WFL_ERR_CUDA; }
        unsigned long long zero = 0;
        CU(cudaMemcpyAsync(&ctr->n_overflow, &zero, sizeof zero, cudaMemcpyHostToDevice, e->stream));
        CU(cudaMemcpyAsync(&ctr->n_fallback2, &zero, sizeof zero, cudaMemcpyHostToDevice, e->stream));
        if ((rc = run_pipeline_list(e, ctr, list, grow))) return rc;
    }
    e->members_total = totals[0];
    if (out) {
        out->members_used = e->members_total;
        if (out->members && out->members_capacity < e->members_total) {
            set_err(e, "members buffer too small: need %lld", (long long)e->members_total);
            e->have_results = true;
            return WFL_ERR_CAPACITY;
        }
        CU(cudaEventElapsedTime(&e->stats.ms_d2h, e->ev[4], e->ev[6]));
    }
    e->stats.matched_pairs = (int64_t)hc.matched_pairs;
    e->stats.groups = (int64_t)hc.groups;
    e->stats.levels = (int64_t)hc.levels;
    e->stats.pairs_tested = (int64_t)hc.pairs_tested;
    e->stats.pairs_scored = (int64_t)hc.pairs_scored;
    e->stats.smem_contigs = (int64_t)hc.smem_contigs;
    e->stats.guard_trips = (int64_t)hc.guard_trips;
    e->stats.refined_groups = (int64_t)hc.refined_groups;
    for (int q = 0; q < 12; ++q) e->stats.phase_cycles[q] = (int64_t)hc.phase_cycles[q];
    CU(cudaEventElapsedTime(&e->stats.ms_score_kernel, e->ev[1], e->ev[2]));
    CU(cudaEventElapsedTime(&e->stats.ms_kernels, e->ev[1], e->ev[3]));
    e->have_results = true;
    return WFL_OK;
}

int run_kernels(wfl_engine *e, bool streamed, wfl_results *out) {
    if (!e->have_params || !e->have_tax || !e->have_batch) {
        set_err(e, "params, taxonomy and batch must be set before running");
        return WFL_ERR_STATE;
    }
    const float h2d = e->stats.ms_h2d;
    e->dt_ready = false;
    e->stats = wfl_stats{};
    e->stats.ms_h2d = h2d;
    e->stats.contigs = e->n;
    e->stats.hits = e->nh;
    e->stats.loci = e->nl;
    for (int round = 0; round < 8; ++round) {
        bool restart = false;
        int rc = run_once(e, streamed, out, &restart);
        if (rc || !restart) return rc;
    }
    set_err(e, "member pool keeps overflowing");
    return WFL_ERR_CUDA;
}

// `host_hits` false: the hit columns are left to the caller (wfl_upload_parsed fills them on the device).
int stage_inputs(wfl_engine *e, const HostBatch &in, bool copy_all, bool host_hits = true) {
    if (!e->have_params || !e->have_tax) {
        set_err(e, "set params and taxonomy before uploading a batch");
        return WFL_ERR_STATE;
    }
    int rc = check_host_batch(e, in);
    if (rc) return rc;
    e->have_batch = e->have_results = false;
    e->n = in.n;
    e->nh = in.nh;
    e->nl = in.nl;
    e->S = e->P.p.n_systems;
    e->packed = in.packed;
    DevBatch &b = e->b;
    b.n_contigs = e->n;
    b.n_hits = e->nh;
    b.n_loci = e->nl;
    const size_t n1 = (size_t)e->n + 1, nh = (size_t)e->nh, nl = (size_t)e->nl;
    e->chunks.clear();
    e->chunks_streamed = false;
    // every fallible allocation first: no H2D copy may be in flight when this function fails (the caller owns the
    // host buffers)
    for (int i = 0; i < in.ncol; ++i)
        if (in.col[i]) {
            void *p;
            if ((rc = outbuf(e, e->in[2 + i], nh * in.esz[i], reinterpret_cast<char **>(&p)))) return rc;
        }
    {
        int32_t *p4;
        int8_t *p1;
        int64_t *p8;
        if ((rc = outbuf(e, e->in[9], nl, &p4)) || (rc = outbuf(e, e->in[10], nl, &p4)) || (rc = outbuf(e, e->in[11], nl, &p1)) ||
            (rc = outbuf(e, e->in[0], n1, &p8)) || (rc = outbuf(e, e->in[1], n1, &p8)))
            return rc;
    }
    {
        int maxlen = 0;
        for (int64_t i = 0; i < in.nl; ++i) {
            int d = in.locus_end[i] - in.locus_start[i];
            d = (d < 0 ? -d : d) + 1;
            maxlen = d > maxlen ? d : maxlen;
        }
        if ((rc = ensure_plan_table(e, maxlen))) return rc;
    }
    bind_device_batch(e);
    b.hit_off = static_cast<const int64_t *>(e->in[0].p);
    b.locus_off = static_cast<const int64_t *>(e->in[1].p);
    // The CSR offsets go first.  Plugin call: on the COPY stream, ahead of chunk 0 (two streams feeding the same DMA
    // queue are not ordered by issue time: on the compute stream they ended up behind the whole bulk transfer and the
    // first kernel with them); chunk 0's event covers them.
    cudaStream_t os = copy_all ? e->stream : e->copy_stream;
    CU(cudaEventRecord(e->ev[0], os));
    CU(cudaMemcpyAsync(e->in[0].p, in.hit_off, n1 * 8, cudaMemcpyHostToDevice, os));
    CU(cudaMemcpyAsync(e->in[1].p, in.locus_off, n1 * 8, cudaMemcpyHostToDevice, os));
    const size_t row = hit_row_bytes(in);
    if (!copy_all) {
        // plugin call: the chunked H2D copies start NOW on the copy stream; the host-side preparation below and the
        // kernels overlap with the transfer
        if (e->n > 0) {
            plan_chunks(e, in.hit_off, in.locus_off, true, row);
            trace("chunks planned");
            if ((rc = issue_chunk_copies(e, in))) { cudaStreamSynchronize(e->copy_stream); return rc; }
            trace("chunk copies issued");
        }
    } else {
        for (int i = 0; i < in.ncol; ++i)
            if (in.col[i] && nh && host_hits)
                CU(cudaMemcpyAsync(dev_col(e, i), in.col[i], nh * in.esz[i], cudaMemcpyHostToDevice, os));
        if (nl) {
            CU(cudaMemcpyAsync(e->in[9].p, in.locus_start, nl * 4, cudaMemcpyHostToDevice, os));
            CU(cudaMemcpyAsync(e->in[10].p, in.locus_end, nl * 4, cudaMemcpyHostToDevice, os));
            CU(cudaMemcpyAsync(e->in[11].p, in.locus_strand, nl, cudaMemcpyHostToDevice, os));
        }
    }
    e->h_hit_off.assign(in.hit_off, in.hit_off + n1);
    e->h_locus_off.assign(in.locus_off, in.locus_off + n1);
    trace("host prep done");
    if (copy_all) {
        CU(cudaEventRecord(e->ev[1], e->stream));
        CU(cudaStreamSynchronize(e->stream));
        CU(cudaEventElapsedTime(&e->stats.ms_h2d, e->ev[0], e->ev[1]));
    } else if (e->n == 0) {
        CU(cudaStreamSynchronize(e->copy_stream));   // no chunk event will order the (empty) offsets
    }
    e->have_batch = true;
    return WFL_OK;
}

int download(wfl_engine *e, wfl_results *out) {
    if (!e->have_results) {
        set_err(e, "no results to download");
        return WFL_ERR_STATE;
    }
    if (!out) { set_err(e, "null results"); return WFL_ERR_ARG; }
    out->members_used = e->members_total;
    if (out->members && out->members_capacity < e->members_total) {
        set_err(e, "members buffer too small: need %lld", (long long)e->members_total);
        return WFL_ERR_CAPACITY;
    }
    int rc;
    CU(cudaEventRecord(e->ev[4], e->stream));
    if ((rc = queue_downloads(e, out, (size_t)e->members_total))) return rc;
    CU(cudaEventRecord(e->ev[6], e->stream));
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaEventElapsedTime(&e->stats.ms_d2h, e->ev[4], e->ev[6]));
    return WFL_OK;
}

int score_host_batch(wfl_engine *e, const HostBatch &hb, wfl_results *out) {
    trace("begin");
    int rc = stage_inputs(e, hb, false);
    if (rc) return rc;
    trace("inputs staged, copies in flight");
    rc = run_kernels(e, true, out);
    if (rc && rc != WFL_ERR_CAPACITY) {
        // the caller owns the host buffers: nothing of ours may still be reading them when we return an error
        cudaStreamSynchronize(e->copy_stream);
        cudaStreamSynchronize(e->stream);
        cudaStreamSynchronize(e->stream2);
        return rc;
    }
    trace("kernels + compaction + downloads done");
    float h2d = 0.f;
    if (e->n > 0 && cudaEventElapsedTime(&h2d, e->ev[0], e->ev[5]) == cudaSuccess) e->stats.ms_h2d = h2d;
    return rc;
}

// ---- results packed into one device buffer (multi-GPU gather) ----
struct PackArgs {
    const void *src[18];
    int64_t off[18], bytes[18];
    char *dst;
    int64_t header[8];
};

__global__ void wfl_pack_results_kernel(const PackArgs a) {
    const int sec = blockIdx.y;
    const int64_t n16 = (a.bytes[sec] + 15) / 16;
    const uint4 *s = static_cast<const uint4 *>(a.src[sec]);
    uint4 *d = reinterpret_cast<uint4 *>(a.dst + a.off[sec]);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t rem = a.bytes[sec] - 16 * i;
        if (rem >= 16) {
            d[i] = s[i];
        } else {   // a section's last, partial chunk: the padding is zero (and nothing past the section is read)
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            const unsigned char *sb = reinterpret_cast<const unsigned char *>(s + i);
            unsigned char *vb = reinterpret_cast<unsigned char *>(&v);
            for (int k = 0; k < (int)rem; ++k) vb[k] = sb[k];
            d[i] = v;
        }
    }
    if (sec == 0 && blockIdx.x == 0 && threadIdx.x < 8) reinterpret_cast<int64_t *>(a.dst)[threadIdx.x] = a.header[threadIdx.x];
}

int64_t results_layout(int64_t n, int64_t nl, int32_t S, int64_t members, int64_t off[18]) {
    const int64_t sz[18] = {n, n, 4 * n, 4 * n, 4 * n, 4 * n, 4 * n, 4 * n, 8 * n, 8 * n, 8 * (n + 1), 4 * n, 4 * members,
                            nl, nl, 4 * nl * S, 8 * 3, 8 * n};
    int64_t o = 64;
    for (int i = 0; i < 18; ++i) {
        off[i] = o;
        o += (sz[i] + 15) & ~int64_t(15);
    }
    return o;
}

// ---- --write-details text (wfl_details.cu) ----
DetTextArgs details_args(wfl_engine *e) {
    DetTextArgs a{};
    a.b = e->b; a.t = e->tax; a.P = e->P;
    a.anc = static_cast<const int *>(e->anc.p);
    a.anc_rows = e->anc_rows;
    a.dc = static_cast<const int32_t *>(e->det[0].p);
    a.di = static_cast<const int32_t *>(e->det[1].p);
    a.dc_clade = static_cast<const int32_t *>(e->det[2].p);
    a.dl = static_cast<const int32_t *>(e->det[3].p);
    a.ds = static_cast<const double *>(e->det[4].p);
    a.seg = static_cast<const DetSeg *>(e->dt_seg.p);
    a.cname = static_cast<const char *>(e->cname.p);
    a.cname_off = static_cast<const int64_t *>(e->cname_off.p);
    a.tname = static_cast<const char *>(e->tname.p);
    a.tname_off = static_cast<const int64_t *>(e->tname_off.p);
    a.seg_bytes = static_cast<long long *>(e->dt_bytes.p);
    a.text_off = static_cast<const long long *>(e->dt_off.p);
    unsigned long long *ctr = static_cast<unsigned long long *>(e->dt_ctr.p);
    a.max_need = ctr;
    a.n_defer = reinterpret_cast<unsigned int *>(ctr + 1);
    a.err = reinterpret_cast<unsigned int *>(ctr + 2);
    a.n_found = reinterpret_cast<unsigned int *>(ctr + 3);
    return a;
}

// The rows kernel over the segments [s0, s1): every warp of the first launch owns a 32 KB scratch slice; segments
// that need more (many hits or groups) go to a second launch whose slices fit the largest of them.  `text` null: the
// length pass (bytes of every segment); otherwise the segments' text at text_off - text_off[s0].
int details_rows(wfl_engine *e, int64_t s0, int64_t s1, char *text) {
    if (s1 <= s0) return WFL_OK;
    int rc;
    const long long slice1 = 32 << 10, warps1 = (long long)e->sm_count * 64;
    const size_t n = (size_t)(s1 - s0);
    int *defer;
    char *scratch;
    if ((rc = outbuf(e, e->dt_defer[0], n, &defer)) || (rc = outbuf(e, e->dt_defer[1], n, &defer)) ||
        (rc = outbuf(e, e->dt_scratch, (size_t)(slice1 * warps1), &scratch)))
        return rc;
    DetTextArgs a = details_args(e);
    a.text = text;
    a.text_base = e->dt_seg_off[(size_t)s0];
    CU(cudaMemsetAsync(e->dt_ctr.p, 0, 2 * sizeof(unsigned long long), e->stream));
    a.s0 = s0; a.n_list = (long long)n; a.list = nullptr;
    a.scratch = scratch; a.slice = slice1;
    a.defer = static_cast<int *>(e->dt_defer[0].p);
    launch_details_rows(a, std::min<long long>(warps1, ((long long)n + 7) & ~7ll), e->stream);
    CU(cudaGetLastError());
    e->stats.kernel_launches++;
    unsigned long long hc[2] = {0, 0};
    CU(cudaMemcpyAsync(hc, e->dt_ctr.p, sizeof hc, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    const long long n_defer = (long long)(hc[1] & 0xffffffffull);
    if (n_defer == 0) return WFL_OK;
    const long long slice2 = ((long long)hc[0] + 255) & ~255ll;
    // whole blocks of 8 warps: every launched warp owns a slice
    const long long warps2 = (std::max<long long>(1, std::min<long long>(n_defer, (1ll << 30) / slice2)) + 7) & ~7ll;
    if ((rc = outbuf(e, e->dt_scratch, (size_t)(slice2 * warps2), &scratch))) return rc;
    a.list = static_cast<const int *>(e->dt_defer[0].p);
    a.n_list = n_defer;
    a.scratch = scratch; a.slice = slice2;
    a.defer = static_cast<int *>(e->dt_defer[1].p);
    launch_details_rows(a, warps2, e->stream);
    CU(cudaGetLastError());
    e->stats.kernel_launches++;
    return WFL_OK;
}

// ---- the scoring batch from a parser's resident hit columns (wfl_resident_batch.cu) ----
constexpr int PARSED_TAX_SLOTS = 1 << 20;   // the parser's distinct-taxon set (wfl_parse.cu)

int upload_parsed(wfl_engine *e, const wfl_parser *p, const wfl_parsed_batch *in, float *ms_kernels) {
    if (p->device != e->device) {
        set_err(e, "the parser is on cuda:%d, the engine on cuda:%d", p->device, e->device);
        return WFL_ERR_ARG;
    }
    if (!p->blast_ok) { set_err(e, "the parser holds no blastout parse without flagged rows"); return WFL_ERR_STATE; }
    if (!e->have_params || !e->have_tax) { set_err(e, "set params and taxonomy before uploading a batch"); return WFL_ERR_STATE; }
    const int S = e->P.p.n_systems;
    HostBatch h;
    h.n = in->n_contigs; h.nh = in->n_hits; h.nl = in->n_loci;
    h.hit_off = in->hit_off; h.locus_off = in->locus_off;
    h.locus_start = in->locus_start; h.locus_end = in->locus_end; h.locus_strand = in->locus_strand;
    // the sources of the wide columns: qstart qend taxon-slot score scov strand on the device, the system map on the host
    const void *c[7] = {p->col[0].p, p->col[1].p, p->col[5].p, p->col[2].p, p->col[3].p, p->col[4].p,
                        S > 0 ? in->sys_perm : nullptr};
    const int z[7] = {4, 4, 4, 8, 8, 1, 4};
    for (int i = 0; i < 7; ++i) { h.col[i] = c[i]; h.esz[i] = z[i]; }
    h.ncol = 7;
    if ((S > 0) != (in->sys_perm != nullptr)) {
        set_err(e, "sys_perm must be given exactly when n_systems > 0");
        return WFL_ERR_ARG;
    }
    int rc = check_host_batch(e, h);
    if (rc) return rc;
    if (h.nh && (!in->hit_src || !in->slot_node)) { set_err(e, "null array in batch"); return WFL_ERR_ARG; }
    for (int64_t k = 0; k < h.n; ++k) {
        const int64_t cnt = h.hit_off[k + 1] - h.hit_off[k];
        if (cnt && (in->hit_src[k] < 0 || in->hit_src[k] > p->n_rows - cnt)) {
            set_err(e, "contig %lld: rows [%lld, %lld) outside the parser's %lld rows", (long long)k,
                    (long long)in->hit_src[k], (long long)(in->hit_src[k] + cnt), (long long)p->n_rows);
            return WFL_ERR_ARG;
        }
    }
    for (int b = 0; S > 0 && b < 64; ++b)
        if (in->sys_perm[b] < -1 || in->sys_perm[b] >= 32) { set_err(e, "sys_perm[%d] out of range", b); return WFL_ERR_ARG; }
    if ((rc = stage_inputs(e, h, true, false))) return rc;
    e->have_batch = false;   // until the hit columns are in place
    const int64_t n = h.n, nh = h.nh;
    // sort plan (host knows every contig's size): contigs whose keys exceed a first-launch slice go to a second launch
    const bool sort = S == 0 && nh > 0;
    const long long slice1 = 32 << 10, warps1 = std::min<long long>((long long)e->sm_count * 64, (n + 7) & ~7ll);
    long long slice2 = 0;
    std::vector<int> big;
    for (int64_t k = 0; sort && k < n; ++k) {
        long long np2 = 1;
        while (np2 < h.hit_off[k + 1] - h.hit_off[k]) np2 <<= 1;
        if (16 * np2 > slice1) { big.push_back((int)k); slice2 = std::max(slice2, 16 * np2); }
    }
    const long long warps2 = big.empty() ? 0 : (std::max<long long>(1, std::min<long long>((long long)big.size(), (1ll << 30) / slice2)) + 7) & ~7ll;
    int64_t *d_src;
    int32_t *d_lut, *d_perm, *d_list = nullptr;
    unsigned long long *d_red;
    char *scratch = nullptr;
    if ((rc = outbuf(e, e->rb_src, (size_t)std::max<int64_t>(n, 1), &d_src)) ||
        (rc = outbuf(e, e->rb_lut, PARSED_TAX_SLOTS, &d_lut)) || (rc = outbuf(e, e->rb_perm, 64, &d_perm)) ||
        (rc = outbuf(e, e->rb_red, 3, &d_red)) ||
        (sort && (rc = outbuf(e, e->rb_scratch, (size_t)std::max(slice1 * warps1, slice2 * warps2), &scratch))) ||
        (!big.empty() && (rc = outbuf(e, e->rb_list, big.size(), &d_list))))
        return rc;
    if (n && in->hit_src) CU(cudaMemcpyAsync(d_src, in->hit_src, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
    if (in->slot_node) CU(cudaMemcpyAsync(d_lut, in->slot_node, (size_t)PARSED_TAX_SLOTS * 4, cudaMemcpyHostToDevice, e->stream));
    if (S > 0) CU(cudaMemcpyAsync(d_perm, in->sys_perm, 64 * 4, cudaMemcpyHostToDevice, e->stream));
    if (!big.empty()) CU(cudaMemcpyAsync(d_list, big.data(), big.size() * 4, cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemsetAsync(d_red, 0, 3 * sizeof(unsigned long long), e->stream));
    // the parse (and anything else queued on the parser's stream) comes first
    CU(cudaEventRecord(e->ev_join, p->stream));
    CU(cudaStreamWaitEvent(e->stream, e->ev_join, 0));
    CU(cudaEventRecord(e->ev[1], e->stream));
    ResBatchArgs a{};
    a.qstart = static_cast<const int32_t *>(p->col[0].p); a.qend = static_cast<const int32_t *>(p->col[1].p);
    a.score = static_cast<const double *>(p->col[2].p); a.scov = static_cast<const double *>(p->col[3].p);
    a.strand = static_cast<const int8_t *>(p->col[4].p); a.tcode = static_cast<const int32_t *>(p->col[5].p);
    a.rawmask = static_cast<const unsigned long long *>(p->col[6].p);
    a.hit_off = e->b.hit_off; a.hit_src = d_src;
    a.n = n; a.nh = nh;
    a.slot_node = d_lut; a.n_slots = PARSED_TAX_SLOTS; a.n_nodes = e->tax.n_nodes;
    a.sys_perm = S > 0 ? d_perm : nullptr;
    a.o_qstart = static_cast<int32_t *>(dev_col(e, 0)); a.o_qend = static_cast<int32_t *>(dev_col(e, 1));
    a.o_taxon = static_cast<int32_t *>(dev_col(e, 2)); a.o_score = static_cast<double *>(dev_col(e, 3));
    a.o_scov = static_cast<double *>(dev_col(e, 4)); a.o_strand = static_cast<int8_t *>(dev_col(e, 5));
    a.o_sysmask = S > 0 ? static_cast<uint32_t *>(dev_col(e, 6)) : nullptr;
    a.red = d_red;
    unsigned long long red[3] = {0, 0, 0};
    if (nh) {
        launch_resident_gather(a, e->sm_count, e->stream);
        CU(cudaGetLastError());
        CU(cudaEventRecord(e->ev[3], e->stream));
        CU(cudaMemcpyAsync(red, d_red, sizeof red, cudaMemcpyDeviceToHost, e->stream));
    }
    CU(cudaStreamSynchronize(e->stream));
    if (red[0]) {
        set_err(e, "%llu hits carry a taxon slot that maps to no taxonomy node", red[0]);
        return WFL_ERR_ARG;
    }
    if (sort) {
        // Batch.sort_hits' choice of key
        int bits_c = 1, bits_t = 1;
        while (bits_c < 63 && (1ll << bits_c) <= n - 1) ++bits_c;
        while (bits_t < 63 && (1ull << bits_t) <= red[2]) ++bits_t;
        const int bits_s = 63 - bits_c - bits_t;
        double smax;
        memcpy(&smax, &red[1], 8);
        a.quantised = bits_s >= 20 && smax > 0.0;
        a.bits_s = bits_s;
        a.smax = smax;
        a.scratch = scratch;
        a.slice = slice1;
        CU(cudaEventRecord(e->ev[4], e->stream));
        launch_resident_sort(a, warps1, e->stream);
        CU(cudaGetLastError());
        if (!big.empty()) {
            a.list = d_list;
            a.n_list = (long long)big.size();
            a.slice = slice2;
            launch_resident_sort(a, warps2, e->stream);
            CU(cudaGetLastError());
        }
    }
    CU(cudaEventRecord(e->ev[2], e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (ms_kernels) {   // the gather, plus the sort when there is one (not the host's wait in between)
        float t = 0.f;
        *ms_kernels = 0.f;
        if (nh) CU(cudaEventElapsedTime(ms_kernels, e->ev[1], e->ev[3]));
        if (sort) CU(cudaEventElapsedTime(&t, e->ev[4], e->ev[2]));
        *ms_kernels += t;
    }
    e->have_batch = true;
    return WFL_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// exported entry points
// ---------------------------------------------------------------------------------------------

extern "C" {

int wfl_abi_version(void) { return WFL_ABI_VERSION; }

int wfl_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int wfl_set_option(wfl_engine *e, const char *name, int64_t value) {
    if (!e || !name) return WFL_ERR_ARG;
    const std::string k(name);
    if (k == "exact") e->exact = value != 0;
    else if (k == "fast_kcap" || k == "fast_hcap") e->fast_hcap = (int)std::max<int64_t>(0, value);
    else if (k == "fast_hscale_pct") e->fast_hscale = std::max<int64_t>(50, value) / 100.0;
    else if (k == "fast_mcap") e->fast_mcap = (int)std::max<int64_t>(0, value);
    else if (k == "fast_tcap") e->fast_tcap = (int)std::max<int64_t>(0, value);
    else if (k == "details") e->det_cap = std::max<int64_t>(0, value);
    else if (k == "fast_passes") e->fast_passes = value >= 2 ? 2 : 1;
    else if (k == "fast_ncap") e->fast_ncap = (int)std::max<int64_t>(0, value);
    else if (k == "pool_mb") e->pipe_pool_bytes = (size_t)std::max<int64_t>(0, value) << 20;
    else if (k == "chunk_mb") { e->chunk_bytes = (size_t)std::max<int64_t>(1, value) << 20; e->chunk_fixed = true; }
    else if (k == "streams") e->n_slots = value >= 2 ? 2 : 1;
    else if (k == "k2_cap") e->k2_cap_override = (size_t)std::max<int64_t>(0, value);
    else { set_err(e, "unknown option %s", name); return WFL_ERR_ARG; }
    e->have_results = false;
    e->cfg_key[0] = -1;
    return WFL_OK;
}

int wfl_create(int device, wfl_engine **out) {
    if (!out) return WFL_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return WFL_ERR_CUDA;
    wfl_engine *e = new wfl_engine();
    e->device = device;
    cudaDeviceProp prop;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess ||
        cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&e->stream2, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess) {
        delete e;
        return WFL_ERR_CUDA;
    }
    e->sm_count = prop.multiProcessorCount;
    e->smem_optin = prop.sharedMemPerBlockOptin;
    // environment twins of wfl_set_option (read once here)
    if (const char *k = getenv("WFL_K2")) e->exact = std::string(k) == "exact";
    if (const char *k = getenv("WFL_K2_CAP")) e->k2_cap_override = (size_t)std::max<long long>(0, atoll(k));
    if (const char *k = getenv("WFL_POOL_MB")) e->pipe_pool_bytes = (size_t)atoll(k) << 20;
    if (const char *k = getenv("WFL_CHUNK_MB")) { e->chunk_bytes = (size_t)std::max<long long>(1, atoll(k)) << 20; e->chunk_fixed = true; }
    if (const char *k = getenv("WFL_STREAMS")) e->n_slots = atoi(k) >= 2 ? 2 : 1;
    if (const char *k = getenv("WFL_FAST_HCAP")) e->fast_hcap = atoi(k);
    if (const char *k = getenv("WFL_FAST_HSCALE")) e->fast_hscale = std::max(0.5, atof(k));
    if (const char *k = getenv("WFL_FAST_TCAP")) e->fast_tcap = atoi(k);
    if (const char *k = getenv("WFL_FAST_NCAP")) e->fast_ncap = atoi(k);
    for (auto &ev : e->ev)
        if (cudaEventCreate(&ev) != cudaSuccess) {
            delete e;
            return WFL_ERR_CUDA;
        }
    *out = e;
    return WFL_OK;
}

void wfl_destroy(wfl_engine *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    auto fr = [](Buf &b) { if (b.p) cudaFree(b.p); b.p = nullptr; };
    for (auto &b : e->tx) fr(b);
    for (auto &b : e->in) fr(b);
    for (auto &b : e->out) fr(b);
    for (auto &b : e->cm) fr(b);
    for (auto &b : e->dbg) fr(b);
    fr(e->anc); fr(e->ctr); fr(e->work); fr(e->scratch); fr(e->plan_index); fr(e->plan_data);
    for (auto &b : e->det) fr(b);
    for (Buf *b : {&e->tname, &e->tname_off, &e->cname, &e->cname_off, &e->dt_found, &e->dt_seg, &e->dt_off, &e->dt_bytes,
                   &e->dt_scratch, &e->dt_defer[0], &e->dt_defer[1], &e->dt_ctr, &e->dt_text})
        fr(*b);
    fr(e->fb_list); fr(e->fast_scratch); fr(e->fast_wq); fr(e->blob); fr(e->status_tmp);
    for (Buf *b : {&e->rb_src, &e->rb_lut, &e->rb_perm, &e->rb_red, &e->rb_list, &e->rb_scratch}) fr(*b);
    for (int q = 0; q < 2; ++q) { fr(e->pipe_pool[q]); fr(e->pipe_lists[q]); fr(e->pipe_cnt[q]); fr(e->pipe_wq[q]); }
    fr(e->pipe_ctg);
    for (int q = 0; q < 2; ++q) { fr(e->k2_desc[q]); fr(e->k2_order[q]); fr(e->k2_keys[q]); fr(e->k2_meta[q]); }
    for (auto &ev : e->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : e->chunk_ev) cudaEventDestroy(ev);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    if (e->stream2) cudaStreamDestroy(e->stream2);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

const char *wfl_last_error(const wfl_engine *e) { return e ? e->err.c_str() : "null engine"; }

int wfl_set_params(wfl_engine *e, const wfl_params *p) {
    if (!e || !p) return WFL_ERR_ARG;
    if (p->n_systems < 0 || p->n_systems > WFL_MAX_SYSTEMS || p->disambiguate_one < 0 || p->disambiguate_one > 1 ||
        p->disambiguate_two < 0 || p->disambiguate_two > 2 || p->weak_loci < 0 || p->weak_loci > 2 ||
        p->ambiguous_threshold < 0 || p->ambiguous_threshold > 2 || p->sister_penalty < 0 ||
        p->sister_penalty > 2 || p->annotation_threshold < 0 || p->annotation_threshold > 2 ||
        p->jump_taxonomy < 0) {
        set_err(e, "parameter out of range");
        return WFL_ERR_ARG;
    }
    DevParams &P = e->P;
    P.p = *p;
    P.min_thr = std::min(p->k1, p->k2);   // waafle_orgscorer.py:338-339
    P.max_thr = std::max(p->k1, p->k2);
    const bool k1_is_min = p->k1 <= p->k2;
    const int sel_min = k1_is_min ? 0 : 1, sel_max = k1_is_min ? 1 : 0;
    const double tri[3] = {1e-6, P.min_thr, P.max_thr};   // off / lenient / strict
    P.ann_thr = tri[p->annotation_threshold];             // :341-346
    P.k_amb = tri[p->ambiguous_threshold];                // :515-516
    P.amb_sel = p->ambiguous_threshold == 0 ? 2 : (p->ambiguous_threshold == 1 ? sel_min : sel_max);
    P.sister_thr = p->sister_penalty == 1 ? P.max_thr : P.min_thr;   // :720-721
    P.sis_sel = p->sister_penalty == 1 ? sel_max : sel_min;
    e->have_params = true;
    e->have_batch = e->have_results = false;
    return WFL_OK;
}

int wfl_set_taxonomy(wfl_engine *e, int32_t n_nodes, const int32_t *parent, const int32_t *depth,
                     const int32_t *leaf_count, const uint8_t *listed, int32_t root_idx, int32_t unknown_idx) {
    if (!e) return WFL_ERR_ARG;
    if (n_nodes <= 0 || !parent || !depth || !leaf_count || !listed || root_idx < 0 || root_idx >= n_nodes ||
        unknown_idx < 0 || unknown_idx >= n_nodes) {
        set_err(e, "bad taxonomy arguments");
        return WFL_ERR_ARG;
    }
    if (parent[root_idx] != root_idx || depth[root_idx] != 0) {
        set_err(e, "root must be its own parent at depth 0");
        return WFL_ERR_ARG;
    }
    int max_depth = 0;
    for (int32_t i = 0; i < n_nodes; ++i) {
        int32_t p = parent[i];
        if (p < 0 || p >= n_nodes || (i != root_idx && depth[i] != depth[p] + 1)) {
            set_err(e, "taxonomy node %d: parent / depth inconsistent", i);
            return WFL_ERR_ARG;
        }
        max_depth = std::max(max_depth, (int)depth[i]);
    }
    CU(cudaSetDevice(e->device));
    int rc;
    if ((rc = upload(e, e->tx[0], parent, (size_t)n_nodes, &e->tax.parent))) return rc;
    if ((rc = upload(e, e->tx[1], depth, (size_t)n_nodes, &e->tax.depth))) return rc;
    if ((rc = upload(e, e->tx[2], leaf_count, (size_t)n_nodes, &e->tax.leaf_count))) return rc;
    if ((rc = upload(e, e->tx[3], listed, (size_t)n_nodes, &e->tax.listed))) return rc;
    // ancestor table of the fast path: row l = l-th ancestor of every node (raise_taxonomy applied l times,
    // waafle_orgscorer.py:431-445 with utils.py:386-387); row max_depth is all root
    {
        const int rows = std::min(max_depth, 63) + 1;
        std::vector<int32_t> anc((size_t)rows * n_nodes);
        for (int32_t i = 0; i < n_nodes; ++i) anc[i] = i;
        for (int l = 1; l < rows; ++l)
            for (int32_t i = 0; i < n_nodes; ++i) anc[(size_t)l * n_nodes + i] = parent[anc[(size_t)(l - 1) * n_nodes + i]];
        const int32_t *d;
        if ((rc = upload(e, e->anc, anc.data(), anc.size(), &d))) return rc;
        CU(cudaStreamSynchronize(e->stream));
        e->anc_rows = rows;
    }
    CU(cudaStreamSynchronize(e->stream));
    e->tax_max_depth = max_depth;
    e->tax.n_nodes = n_nodes;
    e->tax.root = root_idx;
    e->tax.unknown = unknown_idx;
    e->have_tax = true;
    e->have_tnames = e->dt_ready = false;
    e->have_batch = e->have_results = false;
    return WFL_OK;
}

int wfl_upload_batch(wfl_engine *e, const wfl_batch *in) {
    if (!e || !in) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    return stage_inputs(e, host_batch(in, e->P.p.n_systems), true);
}

int wfl_upload_packed(wfl_engine *e, const wfl_packed_batch *in) {
    if (!e || !in) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    return stage_inputs(e, host_batch(in, e->P.p.n_systems), true);
}

int wfl_upload_parsed(wfl_engine *e, const wfl_parser *p, const wfl_parsed_batch *in, float *ms_kernels) {
    if (!e || !p || !in) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    e->have_batch = e->have_results = false;
    const int rc = upload_parsed(e, p, in, ms_kernels);
    if (rc) {
        cudaStreamSynchronize(e->stream);   // nothing of ours reads the caller's arrays after an error
        e->have_batch = e->have_results = false;
    }
    return rc;
}

int wfl_debug_resident_batch(wfl_engine *e, int32_t *qstart, int32_t *qend, int32_t *taxon, double *score, double *scov,
                             int8_t *strand, uint32_t *sysmask) {
    if (!e) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    if (!e->have_batch || e->packed) { set_err(e, "no resident batch in the wide format"); return WFL_ERR_STATE; }
    void *dst[7] = {qstart, qend, taxon, score, scov, strand, e->S > 0 ? sysmask : nullptr};
    const size_t esz[7] = {4, 4, 4, 8, 8, 1, 4};
    for (int i = 0; i < 7; ++i)
        if (dst[i] && e->nh) CU(cudaMemcpyAsync(dst[i], dev_col(e, i), (size_t)e->nh * esz[i], cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return WFL_OK;
}

int wfl_run_resident(wfl_engine *e) {
    if (!e) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    return run_kernels(e, false, nullptr);
}

int wfl_download_results(wfl_engine *e, wfl_results *out) {
    if (!e) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    return download(e, out);
}

int wfl_score_batch(wfl_engine *e, const wfl_batch *in, wfl_results *out) {
    if (!e || !in) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    return score_host_batch(e, host_batch(in, e->P.p.n_systems), out);
}

int wfl_score_packed(wfl_engine *e, const wfl_packed_batch *in, wfl_results *out) {
    if (!e || !in) return WFL_ERR_ARG;
    CU(cudaSetDevice(e->device));
    return score_host_batch(e, host_batch(in, e->P.p.n_systems), out);
}

int64_t wfl_packed_results_layout(int64_t n_contigs, int64_t n_loci, int32_t n_systems, int64_t n_members, int64_t offsets[18]) {
    int64_t tmp[18];
    return results_layout(n_contigs, n_loci, n_systems, n_members, offsets ? offsets : tmp);
}

int wfl_pack_results(wfl_engine *e, void **dev_ptr, int64_t *bytes, void **stream) {
    if (!e || !dev_ptr || !bytes) return WFL_ERR_ARG;
    if (!e->have_results) { set_err(e, "no results to pack"); return WFL_ERR_STATE; }
    CU(cudaSetDevice(e->device));
    PackArgs pa{};
    const int64_t total = results_layout(e->n, e->nl, e->S, e->members_total, pa.off);
    int rc;
    char *blob;
    if ((rc = outbuf(e, e->blob, (size_t)total, &blob))) return rc;
    const DevOut &o = e->o;
    const void *src[18] = {o.call, o.direction, o.lifts, o.clade1, o.clade2, o.lca, o.best1, o.best2, o.crit, o.rank,
                           e->cm[0].p, e->cm[1].p, e->cm[4].p, o.synteny, o.locus_flags, o.ann_winner, e->cm[2].p, e->cm[3].p};
    const int64_t n = e->n, nl = e->nl;
    const int64_t sz[18] = {n, n, 4 * n, 4 * n, 4 * n, 4 * n, 4 * n, 4 * n, 8 * n, 8 * n, 8 * (n + 1), 4 * n, 4 * e->members_total,
                            nl, nl, 4 * nl * e->S, 8 * 3, 8 * n};
    for (int i = 0; i < 18; ++i) { pa.src[i] = src[i]; pa.bytes[i] = sz[i]; }
    pa.dst = blob;
    pa.header[0] = n; pa.header[1] = nl; pa.header[2] = e->S; pa.header[3] = e->members_total;
    wfl_pack_results_kernel<<<dim3(64, 18), 256, 0, e->stream>>>(pa);
    CU(cudaGetLastError());
    e->stats.kernel_launches++;
    *dev_ptr = blob;
    *bytes = total;
    if (stream) *stream = e->stream;
    return WFL_OK;
}

int64_t wfl_download_details(wfl_engine *e, int32_t *contig, int32_t *iteration, int32_t *clade, int32_t *locus, double *score,
                             int64_t capacity) {
    if (!e) return WFL_ERR_ARG;
    if (!e->have_results || e->det_cap <= 0 || !e->det[5].p) { set_err(e, "no details: set option details=<capacity> and run"); return WFL_ERR_STATE; }
    CU(cudaSetDevice(e->device));
    unsigned long long cnt = 0;
    CU(cudaMemcpy(&cnt, e->det[5].p, sizeof cnt, cudaMemcpyDeviceToHost));
    const size_t m = (size_t)std::min<unsigned long long>(cnt, (unsigned long long)std::min<int64_t>(capacity, e->det_cap));
    if (m && contig && iteration && clade && locus && score) {
        CU(cudaMemcpy(contig, e->det[0].p, m * 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(iteration, e->det[1].p, m * 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(clade, e->det[2].p, m * 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(locus, e->det[3].p, m * 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(score, e->det[4].p, m * 8, cudaMemcpyDeviceToHost));
    }
    return (int64_t)cnt;   // entries the run produced (may exceed the capacity: run again with a larger one)
}

int wfl_host_alloc(size_t bytes, void **out) {
    if (!out) return WFL_ERR_ARG;
    *out = nullptr;
    if (cudaHostAlloc(out, bytes ? bytes : 16, cudaHostAllocDefault) != cudaSuccess) return WFL_ERR_CUDA;
    return WFL_OK;
}

void wfl_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

int wfl_get_stats(const wfl_engine *e, wfl_stats *out) {
    if (!e || !out) return WFL_ERR_ARG;
    *out = e->stats;
    return WFL_OK;
}

int64_t wfl_debug_gene_scores(wfl_engine *e, int64_t contig, int32_t *clade, int32_t *locus, double *score,
                              int64_t capacity) {
    if (!e) return WFL_ERR_ARG;
    if (!e->have_batch) { set_err(e, "no resident batch"); return WFL_ERR_STATE; }
    if (contig < 0 || contig >= e->n || capacity < 0) { set_err(e, "bad contig index"); return WFL_ERR_ARG; }
    CU(cudaSetDevice(e->device));
    int rc = alloc_outputs(e);
    if (rc) return rc;
    DevCounters *ctr;
    int32_t *dc, *dl;
    double *ds;
    long long *dn;
    size_t cap = (size_t)std::max<int64_t>(capacity, 1);
    if ((rc = outbuf(e, e->ctr, 1, &ctr)) || (rc = outbuf(e, e->dbg[0], cap, &dc)) ||
        (rc = outbuf(e, e->dbg[1], cap, &dl)) || (rc = outbuf(e, e->dbg[2], cap, &ds)) ||
        (rc = outbuf(e, e->dbg[3], 1, &dn)))
        return rc;
    CU(cudaMemsetAsync(ctr, 0, sizeof(DevCounters), e->stream));
    CU(cudaMemsetAsync(dn, 0, sizeof(long long), e->stream));
    // the exact pipeline over this one contig, with the level-0 dump switched on
    if ((rc = launch_pipeline(e, ctr, nullptr, contig, 1, (size_t)(e->h_hit_off[contig + 1] - e->h_hit_off[contig]), 0, 16, contig)))
        return rc;
    long long cnt = 0;
    CU(cudaMemcpyAsync(&cnt, dn, sizeof cnt, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    size_t m = (size_t)std::min<long long>(cnt, capacity);
    if (m) {
        CU(cudaMemcpy(clade, dc, m * sizeof(int32_t), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(locus, dl, m * sizeof(int32_t), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(score, ds, m * sizeof(double), cudaMemcpyDeviceToHost));
    }
    e->have_results = false;
    return cnt;
}

int wfl_set_clade_names(wfl_engine *e, int32_t n_nodes, const char *blob, const int64_t *off) {
    if (!e) return WFL_ERR_ARG;
    if (!e->have_tax || n_nodes != e->tax.n_nodes) { set_err(e, "clade names need the taxonomy they name"); return WFL_ERR_STATE; }
    if (!off || off[0] != 0 || (off[n_nodes] > 0 && !blob)) { set_err(e, "bad clade name blob"); return WFL_ERR_ARG; }
    for (int32_t i = 0; i < n_nodes; ++i)
        if (off[i + 1] < off[i]) { set_err(e, "clade name offsets are not monotone"); return WFL_ERR_ARG; }
    CU(cudaSetDevice(e->device));
    int rc;
    const char *d1;
    const int64_t *d2;
    if ((rc = upload(e, e->tname, blob, (size_t)off[n_nodes], &d1)) || (rc = upload(e, e->tname_off, off, (size_t)n_nodes + 1, &d2)))
        return rc;
    CU(cudaStreamSynchronize(e->stream));
    e->have_tnames = true;
    return WFL_OK;
}

int64_t wfl_details_prepare(wfl_engine *e, int64_t n_order, const int32_t *order, const char *names, const int64_t *names_off,
                            int64_t *bytes_before, float *ms_kernels) {
    if (!e) return WFL_ERR_ARG;
    e->dt_ready = false;
    if (!e->have_results || e->det_cap <= 0 || !e->det[5].p) { set_err(e, "no details: set option details=<capacity> and run"); return WFL_ERR_STATE; }
    if (!e->have_tnames) { set_err(e, "no clade names: wfl_set_clade_names after wfl_set_taxonomy"); return WFL_ERR_STATE; }
    if (n_order < 0 || (n_order && !order) || !names_off || names_off[0] != 0 || (names_off[e->n] > 0 && !names)) {
        set_err(e, "bad contig order or names");
        return WFL_ERR_ARG;
    }
    std::vector<int64_t> rank((size_t)e->n, -1);
    for (int64_t r = 0; r < n_order; ++r) {
        if (order[r] < 0 || order[r] >= e->n || rank[(size_t)order[r]] >= 0) {
            set_err(e, "contig order: index out of range or repeated at position %lld", (long long)r);
            return WFL_ERR_ARG;
        }
        rank[(size_t)order[r]] = r;
    }
    for (int64_t c = 0; c < e->n; ++c)
        if (names_off[c + 1] < names_off[c]) { set_err(e, "contig name offsets are not monotone"); return WFL_ERR_ARG; }
    CU(cudaSetDevice(e->device));
    unsigned long long cnt = 0;
    CU(cudaMemcpy(&cnt, e->det[5].p, sizeof cnt, cudaMemcpyDeviceToHost));
    if ((long long)cnt > e->det_cap) { set_err(e, "details dump overflowed: run again with details >= %llu", cnt); return WFL_ERR_CAPACITY; }
    int rc;
    const char *d1;
    const int64_t *d2;
    unsigned long long *ctr;
    DetSeg *found;
    if ((rc = upload(e, e->cname, names, (size_t)names_off[e->n], &d1)) ||
        (rc = upload(e, e->cname_off, names_off, (size_t)e->n + 1, &d2)) || (rc = outbuf(e, e->dt_ctr, 4, &ctr)) ||
        (rc = outbuf(e, e->dt_found, (size_t)cnt, &found)))
        return rc;
    CU(cudaEventRecord(e->ev[0], e->stream));
    CU(cudaMemsetAsync(ctr, 0, 4 * sizeof(unsigned long long), e->stream));
    DetTextArgs a = details_args(e);
    a.n_dump = (long long)cnt;
    a.found = found;
    launch_details_segments(a, e->stream);
    CU(cudaGetLastError());
    e->stats.kernel_launches++;
    unsigned long long hc[4];
    CU(cudaMemcpyAsync(hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    const size_t nf = (size_t)(hc[3] & 0xffffffffull);
    std::vector<DetSeg> segs(nf);
    if (nf) CU(cudaMemcpy(segs.data(), found, nf * sizeof(DetSeg), cudaMemcpyDeviceToHost));
    // row order: the caller's contig order, then evaluation index; a replayed contig's second copy of a level goes
    std::vector<DetSeg> keep;
    keep.reserve(nf);
    for (const DetSeg &d : segs)
        if (d.contig >= 0 && d.contig < e->n && rank[(size_t)d.contig] >= 0) keep.push_back(d);
    std::sort(keep.begin(), keep.end(), [&](const DetSeg &x, const DetSeg &y) {
        const int64_t rx = rank[(size_t)x.contig], ry = rank[(size_t)y.contig];
        return rx != ry ? rx < ry : (x.iter != y.iter ? x.iter < y.iter : x.start < y.start);
    });
    keep.erase(std::unique(keep.begin(), keep.end(), [](const DetSeg &x, const DetSeg &y) {
        return x.contig == y.contig && x.iter == y.iter;
    }), keep.end());
    const size_t ns = keep.size();
    DetSeg *dseg;
    long long *dbytes, *doff;
    if ((rc = outbuf(e, e->dt_seg, ns, &dseg)) || (rc = outbuf(e, e->dt_bytes, ns, &dbytes)) || (rc = outbuf(e, e->dt_off, ns, &doff)))
        return rc;
    if (ns) CU(cudaMemcpyAsync(dseg, keep.data(), ns * sizeof(DetSeg), cudaMemcpyHostToDevice, e->stream));
    e->dt_seg_off.assign(ns + 1, 0);
    if ((rc = details_rows(e, 0, (int64_t)ns, nullptr))) return rc;
    std::vector<long long> nb(ns);
    unsigned long long hc2[4];
    CU(cudaMemcpyAsync(hc2, ctr, sizeof hc2, cudaMemcpyDeviceToHost, e->stream));
    if (ns) CU(cudaMemcpyAsync(nb.data(), dbytes, ns * sizeof(long long), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaEventRecord(e->ev[1], e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (hc2[2] & 0xffffffffull) {
        set_err(e, "a gene score lies outside the exactly printable range |x| < 2^53");
        return WFL_ERR_RANGE;
    }
    for (size_t s = 0; s < ns; ++s) e->dt_seg_off[s + 1] = e->dt_seg_off[s] + nb[s];
    if (ns) CU(cudaMemcpyAsync(doff, e->dt_seg_off.data(), ns * sizeof(long long), cudaMemcpyHostToDevice, e->stream));
    e->dt_rank_seg.assign((size_t)n_order + 1, 0);
    size_t s = 0;
    for (int64_t r = 0; r <= n_order; ++r) {
        while (s < ns && rank[(size_t)keep[s].contig] < r) ++s;
        e->dt_rank_seg[(size_t)r] = (int64_t)s;
        if (bytes_before) bytes_before[r] = e->dt_seg_off[s];
    }
    CU(cudaStreamSynchronize(e->stream));
    if (ms_kernels) CU(cudaEventElapsedTime(ms_kernels, e->ev[0], e->ev[1]));
    e->dt_ready = true;
    return e->dt_seg_off[ns];
}

int64_t wfl_details_text(wfl_engine *e, int64_t r0, int64_t r1, char *buf, int64_t capacity, float *ms_kernels,
                         float *ms_d2h) {
    if (!e) return WFL_ERR_ARG;
    if (!e->dt_ready || !e->have_results) { set_err(e, "no prepared details: wfl_details_prepare after a details run"); return WFL_ERR_STATE; }
    const int64_t n_order = (int64_t)e->dt_rank_seg.size() - 1;
    if (r0 < 0 || r1 < r0 || r1 > n_order) { set_err(e, "bad range of the contig order"); return WFL_ERR_ARG; }
    const int64_t s0 = e->dt_rank_seg[(size_t)r0], s1 = e->dt_rank_seg[(size_t)r1];
    const int64_t total = e->dt_seg_off[(size_t)s1] - e->dt_seg_off[(size_t)s0];
    if (!buf || capacity < total) return total;
    CU(cudaSetDevice(e->device));
    int rc;
    char *text;
    if ((rc = outbuf(e, e->dt_text, (size_t)total, &text))) return rc;
    CU(cudaEventRecord(e->ev[0], e->stream));
    if ((rc = details_rows(e, s0, s1, text))) return rc;
    CU(cudaEventRecord(e->ev[1], e->stream));
    if (total) CU(cudaMemcpyAsync(buf, text, (size_t)total, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaEventRecord(e->ev[2], e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (ms_kernels) CU(cudaEventElapsedTime(ms_kernels, e->ev[0], e->ev[1]));
    if (ms_d2h) CU(cudaEventElapsedTime(ms_d2h, e->ev[1], e->ev[2]));
    return total;
}

int64_t wfl_debug_format_scores(wfl_engine *e, const double *x, int64_t n, char *text, int32_t *len) {
    if (!e) return WFL_ERR_ARG;
    if (n < 0 || (n && (!x || !text || !len))) { set_err(e, "bad arguments"); return WFL_ERR_ARG; }
    CU(cudaSetDevice(e->device));
    int rc;
    const double *dx;
    char *dt;
    int *dl;
    unsigned long long *ctr;
    if ((rc = upload(e, e->dbg[2], x, (size_t)n, &dx)) || (rc = outbuf(e, e->dt_text, 24 * (size_t)n, &dt)) ||
        (rc = outbuf(e, e->dbg[0], (size_t)n, &dl)) || (rc = outbuf(e, e->dt_ctr, 4, &ctr)))
        return rc;
    CU(cudaMemsetAsync(ctr, 0, 4 * sizeof(unsigned long long), e->stream));
    if (n) launch_format3(dx, n, dt, dl, reinterpret_cast<unsigned int *>(ctr + 2), e->stream);
    CU(cudaGetLastError());
    unsigned long long hc[4];
    CU(cudaMemcpyAsync(hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, e->stream));
    if (n) {
        CU(cudaMemcpyAsync(text, dt, 24 * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
        CU(cudaMemcpyAsync(len, dl, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    }
    CU(cudaStreamSynchronize(e->stream));
    if (hc[2] & 0xffffffffull) {
        set_err(e, "%u value(s) outside the exactly printable range |x| < 2^53", (unsigned)(hc[2] & 0xffffffffull));
        return WFL_ERR_RANGE;
    }
    return n;
}

}  // extern "C"
