// Front-end parsing on the device (SURVEY 8f rank 1): BLAST outfmt-6 text -> the hit columns the engine consumes.
//
// Replaces the per-row `Hit` objects of waafle/utils.py:192-241 (and iter_contig_hits :255-270): the raw text of a
// blastout file (15 tab-separated fields per row, utils.py:167-183) is shipped to the GPU as is;
//   wfl_parse_lines_*  find the row boundaries (newline count per tile, scan, scatter);
//   wfl_parse_rows     one thread per row: splits the fields, converts the integers and the decimal `pident` exactly
//                      (integer mantissa / power of ten: the correctly rounded double, i.e. what float() returns), and
//                      computes scov_modified and waafle_score in the reference's operation order (utils.py:214-229);
//                      the taxon (sseqid field 1) and the annotation systems (fields 2+, "system=value") are
//                      dictionary-coded against two device hash sets that collect the DISTINCT names of the file;
//                      a change of qseqid against the previous row marks a new contig block (utils.py:258-262);
//   wfl_parse_sysmask  re-orders the annotation-system bits once the host has sorted the distinct system names
//                      (the reference's columns are the sorted systems, waafle_orgscorer.py:824-831).
// Anything the device parser does not reproduce exactly (quoted fields, exponent floats, > 15 significant digits, rows
// with a wrong field count, bad subject headers, zero denominators) flags the row; the host then falls back to the CPU
// reader, which has the reference's error behaviour.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>

#include "waafle_b200.h"
#include "wfl_parser.cuh"

namespace wfl {

namespace {

typedef unsigned long long u64;
typedef unsigned int u32;

constexpr int TILE = 8192;        // bytes per block of the line splitter
constexpr int TPB = 256;          // 32 bytes per thread
constexpr u32 TAX_SLOTS = 1u << 20;
constexpr u32 SYS_SLOTS = 64;
constexpr u64 EMPTY_HASH = 0ull;

struct ParseArgs {
    const char *text;
    long long n_bytes;
    long long *tile_count;        // newlines per tile, then exclusive scan
    long long n_tiles;
    long long *row_start;         // [n_rows + 1]
    long long n_rows;
    // per row outputs
    int32_t *qstart, *qend;
    double *score, *scov;
    int8_t *strand;
    int32_t *tcode;               // slot of the taxon name in the distinct-taxon set
    u64 *rawmask;                 // bit = slot of the annotation system in the distinct-system set (re-ordered later)
    long long *ss_off;            // byte offset of the subject header
    int32_t *ss_len;
    uint8_t *newblock;            // qseqid differs from the previous row's
    long long *q_off;             // byte offset / length of the qseqid (read by the host for block starts only)
    int32_t *q_len;
    // distinct sets (open addressing on a 64-bit FNV-1a hash of the name)
    u64 *tax_hash;                // [TAX_SLOTS]
    long long *tax_off;           // [TAX_SLOTS] one occurrence of the slot's name
    int32_t *tax_len;
    u64 *sys_hash;                // [SYS_SLOTS]
    long long *sys_off;
    int32_t *sys_len;
    int *counters;                // 2: flagged rows, 3: first flagged row (min)
};

__device__ __forceinline__ u64 fnv1a(const char *p, int n) {
    u64 h = 1469598103934665603ull;
    for (int i = 0; i < n; ++i) {
        h ^= (unsigned char)p[i];
        h *= 1099511628211ull;
    }
    return h ? h : 1ull;
}

__global__ void __launch_bounds__(TPB) wfl_parse_lines_count(const ParseArgs a) {
    __shared__ int wsum[TPB / 32];
    const long long base = (long long)blockIdx.x * TILE + (long long)threadIdx.x * 32;
    int cnt = 0;
    for (int i = 0; i < 32; ++i) {
        const long long p = base + i;
        if (p < a.n_bytes && a.text[p] == '\n') ++cnt;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < TPB / 32; ++w) t += wsum[w];
        a.tile_count[blockIdx.x] = t;
    }
}

// single block: exclusive scan of the tile counts in place; tile_count[n_tiles] = total
__global__ void __launch_bounds__(1024) wfl_parse_lines_scan(const ParseArgs a) {
    __shared__ long long part[1024];
    __shared__ long long carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (long long base = 0; base < a.n_tiles; base += 1024) {
        const long long i = base + threadIdx.x;
        const long long v = i < a.n_tiles ? a.tile_count[i] : 0;
        part[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            const long long t = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
            __syncthreads();
            part[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < a.n_tiles) a.tile_count[i] = carry_s + part[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s += part[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) a.tile_count[a.n_tiles] = carry_s;
}

// row r + 1 starts after the r-th newline; row 0 starts at byte 0
__global__ void __launch_bounds__(TPB) wfl_parse_lines_scatter(const ParseArgs a) {
    __shared__ int wsum[TPB / 32];
    const long long base = (long long)blockIdx.x * TILE + (long long)threadIdx.x * 32;
    int cnt = 0;
    for (int i = 0; i < 32; ++i) {
        const long long p = base + i;
        if (p < a.n_bytes && a.text[p] == '\n') ++cnt;
    }
    int inc = cnt;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if ((threadIdx.x & 31) >= o) inc += t;
    }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
    __syncthreads();
    int before = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += wsum[w];
    long long idx = a.tile_count[blockIdx.x] + before + inc - cnt;
    for (int i = 0; i < 32; ++i) {
        const long long p = base + i;
        if (p < a.n_bytes && a.text[p] == '\n') a.row_start[++idx] = p + 1;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) a.row_start[0] = 0;
}

// get-or-insert of a name into a distinct set (open addressing on the 64-bit hash); the code of a name is its SLOT, so
// nobody waits for anybody: the thread that claims a slot also records one occurrence of the name for the host
__device__ int distinct_slot(u64 *hkey, u32 slots, long long *roff, int32_t *rlen, u64 h, long long off, int len) {
    u32 s = (u32)(h ^ (h >> 29)) & (slots - 1);
    for (u32 probe = 0; probe < slots; ++probe) {
        u64 cur = hkey[s];
        if (cur == EMPTY_HASH) {
            const u64 old = atomicCAS(&hkey[s], EMPTY_HASH, h);
            if (old == EMPTY_HASH) {
                roff[s] = off;
                rlen[s] = len;
                return (int)s;
            }
            cur = old;
        }
        if (cur == h) return (int)s;
        s = (s + 1) & (slots - 1);
    }
    return -1;
}

__device__ __forceinline__ bool parse_int(const char *p, int n, long long &out) {
    if (n <= 0 || n > 18) return false;
    long long v = 0;
    for (int i = 0; i < n; ++i) {
        const int d = p[i] - '0';
        if (d < 0 || d > 9) return false;
        v = v * 10 + d;
    }
    out = v;
    return true;
}

// digits[.digits] with <= 15 significant digits: mantissa / 10^k is the correctly rounded double
__device__ __forceinline__ bool parse_decimal(const char *p, int n, double &out) {
    if (n <= 0) return false;
    long long m = 0;
    int nd = 0, frac = 0;
    bool dot = false, any = false;
    for (int i = 0; i < n; ++i) {
        const char ch = p[i];
        if (ch == '.') {
            if (dot) return false;
            dot = true;
            continue;
        }
        const int d = ch - '0';
        if (d < 0 || d > 9) return false;
        any = true;
        if (m != 0 || d != 0) ++nd;
        if (nd > 15) return false;
        m = m * 10 + d;
        if (dot) ++frac;
    }
    if (!any || frac > 22) return false;
    double den = 1.0;
    for (int i = 0; i < frac; ++i) den *= 10.0;   // exact up to 10^22
    out = (double)m / den;
    return true;
}

__global__ void __launch_bounds__(128) wfl_parse_rows(const ParseArgs a) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.n_rows) return;
    const long long s = a.row_start[r];
    long long e = a.row_start[r + 1] - 1;               // position of the newline (or n_bytes for an unterminated last row)
    if (r + 1 == a.n_rows && (e < 0 || e >= a.n_bytes || a.text[e] != '\n')) e = a.n_bytes;
    if (e > s && a.text[e - 1] == '\r') --e;
    const char *row = a.text + s;
    const int len = (int)(e - s);
    // field boundaries
    int fs[16], nf = 0;
    fs[0] = 0;
    bool bad = len <= 0;
    for (int i = 0; i < len; ++i) {
        const char ch = row[i];
        if (ch == '\t') {
            if (nf < 15) fs[++nf] = i + 1; else bad = true;
        } else if (ch == '"') {
            bad = true;   // csv quoting: host reader
        }
    }
    ++nf;
    fs[nf < 16 ? nf : 15] = len + 1;
    if (nf != 15) bad = true;   // utils.py:208-209
    long long qlen = 0, slen = 0, alen = 0, qs = 0, qe = 0, ss = 0, se = 0, pos = 0, gaps = 0;
    double pident = 0.0;
    bool minus = false;
    if (!bad) {
#define FIELD(k) (row + fs[k]), (fs[(k) + 1] - fs[k] - 1)
        bad |= !parse_int(FIELD(2), qlen) || !parse_int(FIELD(3), slen) || !parse_int(FIELD(4), alen) ||
               !parse_int(FIELD(5), qs) || !parse_int(FIELD(6), qe) || !parse_int(FIELD(7), ss) ||
               !parse_int(FIELD(8), se) || !parse_decimal(FIELD(9), pident) || !parse_int(FIELD(10), pos) ||
               !parse_int(FIELD(11), gaps);
        const int sl = fs[15] - fs[14] - 1;
        minus = sl == 5 && row[fs[14]] == 'm' && row[fs[14] + 1] == 'i' && row[fs[14] + 2] == 'n' &&
                row[fs[14] + 3] == 'u' && row[fs[14] + 4] == 's';   // utils.py:214
        if (sl == 0 || fs[1] - fs[0] - 1 <= 0) bad = true;
#undef FIELD
    }
    double scov = 0.0, score = 0.0;
    int tcode = -1;
    u64 mask = 0;
    const int q_len = bad ? 0 : fs[1] - fs[0] - 1;
    const int h_off = bad ? 0 : fs[1], h_len = bad ? 0 : fs[2] - fs[1] - 1;
    if (!bad) {
        // utils.py:219-229, same operation order
        const long long s1 = minus ? slen - ss + 1 : ss, s2 = minus ? slen - se + 1 : se;
        const long long ltrim = max(0ll, s1 - qs), rtrim = max(0ll, slen - s1 - qlen + qs);
        const long long den = slen - ltrim - rtrim;
        if (den == 0 || qs > 2147483647ll || qe > 2147483647ll) {
            bad = true;
        } else {
            scov = (double)(s2 - s1 + 1) / (double)den;
            score = scov * pident / 100.0;
        }
        // subject header: geneid|taxon|system=value...   utils.py:231-241
        const char *hp = row + h_off;
        int bar1 = -1, bar2 = -1;
        for (int i = 0; i < h_len && bar2 < 0; ++i)
            if (hp[i] == '|') { if (bar1 < 0) bar1 = i; else bar2 = i; }
        if (bar1 < 0) {
            bad = true;   // "bad subject id header"
        } else {
            const int t0 = bar1 + 1, t1 = bar2 < 0 ? h_len : bar2;
            tcode = distinct_slot(a.tax_hash, TAX_SLOTS, a.tax_off, a.tax_len, fnv1a(hp + t0, t1 - t0), s + h_off + t0, t1 - t0);
            if (tcode < 0) bad = true;
            int i0 = bar2 < 0 ? h_len : bar2 + 1;
            while (i0 <= h_len && bar2 >= 0 && !bad) {   // annotation items
                int i1 = i0, eq = -1, neq = 0;
                while (i1 < h_len && hp[i1] != '|') {
                    if (hp[i1] == '=') { if (eq < 0) eq = i1; ++neq; }
                    ++i1;
                }
                if (neq != 1) { bad = true; break; }   // `system, name = k.split("=")` raises otherwise
                const int sc = distinct_slot(a.sys_hash, SYS_SLOTS, a.sys_off, a.sys_len, fnv1a(hp + i0, eq - i0), s + h_off + i0, eq - i0);
                if (sc < 0) { bad = true; break; }
                mask |= 1ull << sc;
                i0 = i1 + 1;
                if (i1 >= h_len) break;
            }
        }
    }
    if (bad) {
        atomicAdd(&a.counters[2], 1);
        atomicMin(&a.counters[3], (int)min(r, 2147483647ll));
    }
    a.qstart[r] = (int32_t)qs;
    a.qend[r] = (int32_t)qe;
    a.score[r] = score;
    a.scov[r] = scov;
    a.strand[r] = minus ? '-' : '+';
    a.tcode[r] = tcode;
    a.rawmask[r] = mask;
    a.ss_off[r] = s + h_off;
    a.ss_len[r] = h_len;
    a.q_off[r] = s;
    a.q_len[r] = q_len;
    // new contig block: the qseqid differs from the previous row's
    bool nb = r == 0;
    if (r > 0 && !bad) {
        const long long ps = a.row_start[r - 1];
        int pl = 0;
        while (ps + pl < s && a.text[ps + pl] != '\t' && a.text[ps + pl] != '\n') ++pl;
        nb = pl != q_len;
        for (int i = 0; i < q_len && !nb; ++i) nb = a.text[ps + i] != row[i];
    }
    a.newblock[r] = nb ? 1 : 0;
}

// perm[slot] = bit of that system in the SORTED system list (-1: not a system)
__global__ void wfl_parse_sysmask(const u64 *raw, uint32_t *mask, long long n, const int *perm) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        u64 m = raw[i];
        u32 out = 0;
        while (m) {
            const int b = __ffsll((long long)m) - 1;
            m &= m - 1;
            if (perm[b] >= 0) out |= 1u << perm[b];
        }
        mask[i] = out;
    }
}

// ---- GFF rows (waafle/utils.py:298-355): seqname, start, end, strand of every locus ------------------------------
struct GffArgs {
    const char *text;
    long long n_bytes;
    const long long *row_start;   // [n_rows + 1]
    long long n_rows;
    int32_t *start, *end;
    int8_t *strand;
    uint8_t *skip;                // comment ('#') or empty row
    uint8_t *newblock;            // seqname differs from the previous locus row's (iter_contig_loci :341-355)
    long long *s_off;
    int32_t *s_len;
    int *counters;                // 2: flagged rows, 3: first flagged row
};

__device__ __forceinline__ void gff_row_span(const GffArgs &a, long long r, long long &s, long long &e) {
    s = a.row_start[r];
    e = a.row_start[r + 1] - 1;                       // position of the newline (or one past the text)
    if (e > a.n_bytes) e = a.n_bytes;
    if (e > s && a.text[e - 1] == '\r') --e;          // csv.excel_tab rows end in CRLF (the reference writes them so)
}

__global__ void __launch_bounds__(128) wfl_parse_gff_rows(const GffArgs a) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.n_rows) return;
    long long s, e;
    gff_row_span(a, r, s, e);
    const bool skip = e <= s || a.text[s] == '#';     // :345-346 (an empty row is not a locus either)
    a.skip[r] = skip ? 1 : 0;
    a.newblock[r] = 0;
    a.start[r] = a.end[r] = 0;
    a.strand[r] = '?';
    a.s_off[r] = s;
    a.s_len[r] = 0;
    if (skip) return;
    // 9 tab-separated fields (:302-303); a field that opens with a quote is left to the CPU reader (csv quoting)
    long long f0[9], f1[9];
    int nf = 0;
    long long b = s;
    bool bad = false;
    for (long long p = s; p <= e; ++p) {
        if (p == e || a.text[p] == '\t') {
            if (nf < 9) { f0[nf] = b; f1[nf] = p; }
            ++nf;
            if (b < e && a.text[b] == '"') bad = true;
            b = p + 1;
        }
    }
    long long v0 = 0, v1 = 0;
    if (nf != 9) bad = true;
    if (!bad) {
        bad = !parse_int(a.text + f0[3], (int)(f1[3] - f0[3]), v0) || !parse_int(a.text + f0[4], (int)(f1[4] - f0[4]), v1) ||
              v0 > 2147483647ll || v1 > 2147483647ll || f1[6] - f0[6] != 1 || f1[0] - f0[0] <= 0 || f1[0] - f0[0] > 2147483647ll;
    }
    if (bad) {
        atomicAdd(&a.counters[2], 1);
        atomicMin(&a.counters[3], (int)(r > 2147483647ll ? 2147483647ll : r));
        return;
    }
    a.start[r] = (int32_t)v0;
    a.end[r] = (int32_t)v1;
    a.strand[r] = (int8_t)a.text[f0[6]];
    a.s_off[r] = f0[0];
    a.s_len[r] = (int32_t)(f1[0] - f0[0]);
    // contig block start: the previous locus row (comments skipped) names another sequence
    long long q = r - 1;
    bool nb = true;
    while (q >= 0) {
        long long qs, qe;
        gff_row_span(a, q, qs, qe);
        if (qe > qs && a.text[qs] != '#') {
            long long t = qs;
            while (t < qe && a.text[t] != '\t') ++t;
            const long long len = t - qs;
            nb = len != f1[0] - f0[0];
            for (long long i = 0; !nb && i < len; ++i) nb = a.text[qs + i] != a.text[f0[0] + i];
            break;
        }
        --q;
    }
    a.newblock[r] = nb ? 1 : 0;
}

}  // namespace

int pensure(wfl_parser *p, PBuf &b, size_t bytes) {
    bytes = (bytes + 255) & ~size_t(255);
    if (bytes == 0) bytes = 256;
    if (b.cap >= bytes) return WFL_OK;
    if (b.p) PCU(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    PCU(cudaMalloc(&b.p, bytes + bytes / 8));
    b.cap = bytes + bytes / 8;
    return WFL_OK;
}

}  // namespace wfl

using namespace wfl;

extern "C" {

int wfl_parser_create(int device, wfl_parser **out) {
    if (!out) return WFL_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return WFL_ERR_CUDA;
    wfl_parser *p = new wfl_parser();
    p->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete p;
        return WFL_ERR_CUDA;
    }
    for (auto &e : p->ev)
        if (cudaEventCreate(&e) != cudaSuccess) { delete p; return WFL_ERR_CUDA; }
    *out = p;
    return WFL_OK;
}

void wfl_parser_destroy(wfl_parser *p) {
    if (!p) return;
    cudaSetDevice(p->device);
    PBuf *all[] = {&p->text, &p->tiles, &p->rows, &p->tax_hash, &p->tax_off, &p->tax_len, &p->sys_hash,
                   &p->sys_off, &p->sys_len, &p->counters, &p->perm, &p->comp, &p->mtab};
    for (PBuf *b : all) if (b->p) cudaFree(b->p);
    for (auto &b : p->col) if (b.p) cudaFree(b.p);
    for (auto &b : p->gcol) if (b.p) cudaFree(b.p);
    if (p->gc_pool.p) cudaFree(p->gc_pool.p);
    for (auto &e : p->ev) if (e) cudaEventDestroy(e);
    if (p->stream) cudaStreamDestroy(p->stream);
    delete p;
}

const char *wfl_parser_last_error(const wfl_parser *p) { return p ? p->err : "null parser"; }

}  // extern "C"

namespace {

// the parse buffers whose size the text alone decides (a no-op when they are large enough)
int parse_buffers(wfl_parser *p, long long n_bytes) {
    int rc;
    const long long n_tiles = (n_bytes + TILE - 1) / TILE;
    if ((rc = pensure(p, p->tiles, (size_t)(n_tiles + 1) * 8)) || (rc = pensure(p, p->tax_hash, (size_t)TAX_SLOTS * 8)) ||
        (rc = pensure(p, p->tax_off, (size_t)TAX_SLOTS * 8)) || (rc = pensure(p, p->tax_len, (size_t)TAX_SLOTS * 4)) ||
        (rc = pensure(p, p->sys_hash, SYS_SLOTS * 8)) || (rc = pensure(p, p->sys_off, SYS_SLOTS * 8)) ||
        (rc = pensure(p, p->sys_len, SYS_SLOTS * 4)) || (rc = pensure(p, p->counters, 16)) ||
        (rc = pensure(p, p->perm, SYS_SLOTS * 4)))
        return rc;
    return WFL_OK;
}

// parse bytes [off, off + n_bytes) of the resident text.  `host_text`: the same bytes on the host when the caller has just
// uploaded them (it recorded ev[0] before the copy), else NULL: the one byte the host needs then comes from the device.
int64_t parse_resident(wfl_parser *p, long long off, long long n_bytes, int32_t *flagged, int64_t *first_flagged,
                       const char *host_text) {
    p->n_bytes = n_bytes;
    p->n_rows = 0;
    p->blast_ok = p->genes_ok = false;
    if (flagged) *flagged = 0;
    if (first_flagged) *first_flagged = -1;
    if (n_bytes == 0) {
        p->blast_ok = true;
        return 0;
    }
    int rc;
    const long long n_tiles = (n_bytes + TILE - 1) / TILE;
    if ((rc = parse_buffers(p, n_bytes))) return rc;
    PCU(cudaEventRecord(p->ev[1], p->stream));
    PCU(cudaMemsetAsync(p->tax_hash.p, 0, (size_t)TAX_SLOTS * 8, p->stream));
    PCU(cudaMemsetAsync(p->sys_hash.p, 0, SYS_SLOTS * 8, p->stream));
    const int init[4] = {0, 0, 0, 2147483647};
    PCU(cudaMemcpyAsync(p->counters.p, init, sizeof init, cudaMemcpyHostToDevice, p->stream));
    ParseArgs a{};
    a.text = static_cast<const char *>(p->text.p) + off;
    a.n_bytes = n_bytes;
    a.tile_count = static_cast<long long *>(p->tiles.p);
    a.n_tiles = n_tiles;
    wfl_parse_lines_count<<<(unsigned)n_tiles, TPB, 0, p->stream>>>(a);
    wfl_parse_lines_scan<<<1, 1024, 0, p->stream>>>(a);
    long long n_newlines = 0;
    char last = host_text ? host_text[n_bytes - 1] : 0;
    PCU(cudaMemcpyAsync(&n_newlines, a.tile_count + n_tiles, 8, cudaMemcpyDeviceToHost, p->stream));
    if (!host_text) PCU(cudaMemcpyAsync(&last, a.text + n_bytes - 1, 1, cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    const bool unterminated = last != '\n';
    const long long n_rows = n_newlines + (unterminated ? 1 : 0);
    p->n_rows = n_rows;
    if ((rc = pensure(p, p->rows, (size_t)(n_rows + 2) * 8))) return rc;
    const size_t esz[13] = {4, 4, 8, 8, 1, 4, 8, 8, 4, 1, 8, 4, 4};
    for (int i = 0; i < 13; ++i)
        if ((rc = pensure(p, p->col[i], (size_t)n_rows * esz[i]))) return rc;
    a.row_start = static_cast<long long *>(p->rows.p);
    a.n_rows = n_rows;
    a.qstart = static_cast<int32_t *>(p->col[0].p); a.qend = static_cast<int32_t *>(p->col[1].p);
    a.score = static_cast<double *>(p->col[2].p); a.scov = static_cast<double *>(p->col[3].p);
    a.strand = static_cast<int8_t *>(p->col[4].p); a.tcode = static_cast<int32_t *>(p->col[5].p);
    a.rawmask = static_cast<u64 *>(p->col[6].p); a.ss_off = static_cast<long long *>(p->col[7].p);
    a.ss_len = static_cast<int32_t *>(p->col[8].p); a.newblock = static_cast<uint8_t *>(p->col[9].p);
    a.q_off = static_cast<long long *>(p->col[10].p); a.q_len = static_cast<int32_t *>(p->col[11].p);
    a.tax_hash = static_cast<u64 *>(p->tax_hash.p);
    a.tax_off = static_cast<long long *>(p->tax_off.p); a.tax_len = static_cast<int32_t *>(p->tax_len.p);
    a.sys_hash = static_cast<u64 *>(p->sys_hash.p);
    a.sys_off = static_cast<long long *>(p->sys_off.p); a.sys_len = static_cast<int32_t *>(p->sys_len.p);
    a.counters = static_cast<int *>(p->counters.p);
    wfl_parse_lines_scatter<<<(unsigned)n_tiles, TPB, 0, p->stream>>>(a);
    if (unterminated) {
        const long long endpos = n_bytes + 1;   // row_start[n_rows] - 1 == n_bytes
        PCU(cudaMemcpyAsync(a.row_start + n_rows, &endpos, 8, cudaMemcpyHostToDevice, p->stream));
    }
    if (n_rows > 0) wfl_parse_rows<<<(unsigned)((n_rows + 127) / 128), 128, 0, p->stream>>>(a);
    PCU(cudaGetLastError());
    PCU(cudaEventRecord(p->ev[2], p->stream));
    int counters[4];
    PCU(cudaMemcpyAsync(counters, p->counters.p, sizeof counters, cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    p->ms_h2d = 0;
    if (host_text) PCU(cudaEventElapsedTime(&p->ms_h2d, p->ev[0], p->ev[1]));
    PCU(cudaEventElapsedTime(&p->ms_kernels, p->ev[1], p->ev[2]));
    if (flagged) *flagged = counters[2];
    if (first_flagged) *first_flagged = counters[2] ? counters[3] : -1;
    p->blast_ok = counters[2] == 0;
    return n_rows;
}

}  // namespace

extern "C" {

/* Ship `n_bytes` of blastout text (whole rows; the caller owns the buffer) and parse it on the device.  Returns the
 * number of rows (>= 0) or a negative wfl_status; *flagged = rows the device parser cannot reproduce exactly (then
 * *first_flagged is the first such row and the caller must use the CPU reader). */
int64_t wfl_parse_blast(wfl_parser *p, const char *text, int64_t n_bytes, int32_t *flagged, int64_t *first_flagged) {
    if (!p || (!text && n_bytes) || n_bytes < 0) return WFL_ERR_ARG;
    PCU(cudaSetDevice(p->device));
    p->text_bytes = 0;
    if (n_bytes > 0) {
        int rc;
        if ((rc = pensure(p, p->text, (size_t)n_bytes + 64)) || (rc = parse_buffers(p, n_bytes))) return rc;
        PCU(cudaEventRecord(p->ev[0], p->stream));
        PCU(cudaMemcpyAsync(p->text.p, text, (size_t)n_bytes, cudaMemcpyHostToDevice, p->stream));
        p->text_bytes = n_bytes;
    }
    return parse_resident(p, 0, n_bytes, flagged, first_flagged, text);
}

/* Parse bytes [off, off + n_bytes) of the resident text (an upload or a BGZF inflate); offsets relative to `off`. */
int64_t wfl_parse_blast_resident(wfl_parser *p, int64_t off, int64_t n_bytes, int32_t *flagged, int64_t *first_flagged) {
    if (!p || off < 0 || n_bytes < 0 || off > p->text_bytes - n_bytes) return WFL_ERR_ARG;
    PCU(cudaSetDevice(p->device));
    return parse_resident(p, off, n_bytes, flagged, first_flagged, nullptr);
}

/* Resident text [off, off + n_bytes) to the host. */
int wfl_parser_text(wfl_parser *p, int64_t off, int64_t n_bytes, char *dst) {
    if (!p || off < 0 || n_bytes < 0 || off > p->text_bytes - n_bytes || (!dst && n_bytes)) return WFL_ERR_ARG;
    if (n_bytes == 0) return WFL_OK;
    PCU(cudaSetDevice(p->device));
    PCU(cudaMemcpyAsync(dst, static_cast<const char *>(p->text.p) + off, (size_t)n_bytes, cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    return WFL_OK;
}

/* The distinct-name sets of the last parse: kind 0 = taxa (2^20 slots), 1 = annotation systems (64 slots).  hash[s] != 0
 * marks an occupied slot; (off[s], len[s]) is one occurrence of its name in the text.  Arrays of `slots` entries. */
int wfl_parse_distinct(wfl_parser *p, int kind, uint64_t *hash, int64_t *off, int32_t *len, int32_t slots) {
    if (!p || !hash || !off || !len) return WFL_ERR_ARG;
    PCU(cudaSetDevice(p->device));
    const int want = kind == 0 ? (int)TAX_SLOTS : (int)SYS_SLOTS;
    if (slots != want) return WFL_ERR_ARG;
    if (p->n_rows == 0) { memset(hash, 0, (size_t)slots * 8); return WFL_OK; }
    PCU(cudaMemcpy(hash, kind == 0 ? p->tax_hash.p : p->sys_hash.p, (size_t)slots * 8, cudaMemcpyDeviceToHost));
    PCU(cudaMemcpy(off, kind == 0 ? p->tax_off.p : p->sys_off.p, (size_t)slots * 8, cudaMemcpyDeviceToHost));
    PCU(cudaMemcpy(len, kind == 0 ? p->tax_len.p : p->sys_len.p, (size_t)slots * 4, cudaMemcpyDeviceToHost));
    return WFL_OK;
}

/* Final step: sys_perm[slot] = bit of that system in the SORTED system list, -1 for empty slots (64 entries; the host read
 * the names with wfl_parse_distinct); then every column is copied to the caller's arrays (each [n_rows]; NULL = skip).
 * tcode[r] is the taxon's slot in the distinct-taxon set. */
int wfl_parse_fetch(wfl_parser *p, const int32_t *sys_perm, int32_t *qstart, int32_t *qend, double *score, double *scov,
                    int8_t *strand, int32_t *tcode, uint32_t *sysmask, int64_t *ss_off, int32_t *ss_len, uint8_t *newblock,
                    int64_t *q_off, int32_t *q_len) {
    if (!p) return WFL_ERR_ARG;
    PCU(cudaSetDevice(p->device));
    const long long n = p->n_rows;
    if (n == 0) return WFL_OK;
    PCU(cudaEventRecord(p->ev[0], p->stream));
    if (sysmask) {
        int32_t none[SYS_SLOTS];
        for (u32 i = 0; i < SYS_SLOTS; ++i) none[i] = -1;
        PCU(cudaMemcpyAsync(p->perm.p, sys_perm ? sys_perm : none, SYS_SLOTS * 4, cudaMemcpyHostToDevice, p->stream));
        wfl_parse_sysmask<<<1024, 256, 0, p->stream>>>(static_cast<const u64 *>(p->col[6].p), static_cast<uint32_t *>(p->col[12].p), n,
                                                       static_cast<const int *>(p->perm.p));
        PCU(cudaGetLastError());
    }
    void *dst[12] = {qstart, qend, score, scov, strand, tcode, sysmask, ss_off, ss_len, newblock, q_off, q_len};
    const int srcc[12] = {0, 1, 2, 3, 4, 5, 12, 7, 8, 9, 10, 11};
    const size_t esz[12] = {4, 4, 8, 8, 1, 4, 4, 8, 4, 1, 8, 4};
    for (int i = 0; i < 12; ++i)
        if (dst[i]) PCU(cudaMemcpyAsync(dst[i], p->col[srcc[i]].p, (size_t)n * esz[i], cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaEventRecord(p->ev[1], p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    PCU(cudaEventElapsedTime(&p->ms_d2h, p->ev[0], p->ev[1]));
    return WFL_OK;
}

/* GFF text (waafle_genecaller / Prodigal style) parsed on the device: replaces the per-row Locus objects of
 * waafle/utils.py:298-355.  Returns the number of text rows (comment and empty rows included: they come back with skip = 1)
 * or a negative wfl_status; *flagged = rows the device does not reproduce (field count, non-integer coordinates, a quoted
 * field, a strand longer than one character): the caller must then use its CPU reader. */
int64_t wfl_parse_gff(wfl_parser *p, const char *text, int64_t n_bytes, int32_t *flagged, int64_t *first_flagged) {
    if (!p || (!text && n_bytes) || n_bytes < 0) return WFL_ERR_ARG;
    PCU(cudaSetDevice(p->device));
    p->gff_rows = 0;
    p->text_bytes = 0;   // the text buffer now holds the GFF
    if (flagged) *flagged = 0;
    if (first_flagged) *first_flagged = -1;
    if (n_bytes == 0) return 0;
    int rc;
    const long long n_tiles = (n_bytes + TILE - 1) / TILE;
    if ((rc = pensure(p, p->text, (size_t)n_bytes + 64)) || (rc = pensure(p, p->tiles, (size_t)(n_tiles + 1) * 8)) ||
        (rc = pensure(p, p->counters, 16)))
        return rc;
    PCU(cudaEventRecord(p->ev[0], p->stream));
    PCU(cudaMemcpyAsync(p->text.p, text, (size_t)n_bytes, cudaMemcpyHostToDevice, p->stream));
    PCU(cudaEventRecord(p->ev[1], p->stream));
    const int init[4] = {0, 0, 0, 2147483647};
    PCU(cudaMemcpyAsync(p->counters.p, init, sizeof init, cudaMemcpyHostToDevice, p->stream));
    ParseArgs a{};
    a.text = static_cast<const char *>(p->text.p);
    a.n_bytes = n_bytes;
    a.tile_count = static_cast<long long *>(p->tiles.p);
    a.n_tiles = n_tiles;
    wfl_parse_lines_count<<<(unsigned)n_tiles, TPB, 0, p->stream>>>(a);
    wfl_parse_lines_scan<<<1, 1024, 0, p->stream>>>(a);
    long long n_newlines = 0;
    PCU(cudaMemcpyAsync(&n_newlines, a.tile_count + n_tiles, 8, cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    const bool unterminated = text[n_bytes - 1] != '\n';
    const long long n_rows = n_newlines + (unterminated ? 1 : 0);
    p->gff_rows = n_rows;
    if ((rc = pensure(p, p->rows, (size_t)(n_rows + 2) * 8))) return rc;
    const size_t esz[7] = {4, 4, 1, 1, 1, 8, 4};
    for (int i = 0; i < 7; ++i)
        if ((rc = pensure(p, p->gcol[i], (size_t)n_rows * esz[i]))) return rc;
    a.row_start = static_cast<long long *>(p->rows.p);
    a.n_rows = n_rows;
    wfl_parse_lines_scatter<<<(unsigned)n_tiles, TPB, 0, p->stream>>>(a);
    if (unterminated) {
        const long long endpos = n_bytes + 1;
        PCU(cudaMemcpyAsync(a.row_start + n_rows, &endpos, 8, cudaMemcpyHostToDevice, p->stream));
    }
    GffArgs g{};
    g.text = a.text; g.n_bytes = n_bytes; g.row_start = a.row_start; g.n_rows = n_rows;
    g.start = static_cast<int32_t *>(p->gcol[0].p); g.end = static_cast<int32_t *>(p->gcol[1].p);
    g.strand = static_cast<int8_t *>(p->gcol[2].p); g.skip = static_cast<uint8_t *>(p->gcol[3].p);
    g.newblock = static_cast<uint8_t *>(p->gcol[4].p); g.s_off = static_cast<long long *>(p->gcol[5].p);
    g.s_len = static_cast<int32_t *>(p->gcol[6].p); g.counters = static_cast<int *>(p->counters.p);
    if (n_rows > 0) wfl_parse_gff_rows<<<(unsigned)((n_rows + 127) / 128), 128, 0, p->stream>>>(g);
    PCU(cudaGetLastError());
    PCU(cudaEventRecord(p->ev[2], p->stream));
    int counters[4];
    PCU(cudaMemcpyAsync(counters, p->counters.p, sizeof counters, cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    PCU(cudaEventElapsedTime(&p->ms_h2d, p->ev[0], p->ev[1]));
    PCU(cudaEventElapsedTime(&p->ms_kernels, p->ev[1], p->ev[2]));
    if (flagged) *flagged = counters[2];
    if (first_flagged) *first_flagged = counters[2] ? counters[3] : -1;
    return n_rows;
}

/* The columns of the last wfl_parse_gff, each [n_rows] (NULL = skip). */
int wfl_parse_gff_fetch(wfl_parser *p, int32_t *start, int32_t *end, int8_t *strand, uint8_t *skip, uint8_t *newblock,
                        int64_t *s_off, int32_t *s_len) {
    if (!p) return WFL_ERR_ARG;
    PCU(cudaSetDevice(p->device));
    const long long n = p->gff_rows;
    if (n == 0) return WFL_OK;
    void *dst[7] = {start, end, strand, skip, newblock, s_off, s_len};
    const size_t esz[7] = {4, 4, 1, 1, 1, 8, 4};
    PCU(cudaEventRecord(p->ev[0], p->stream));
    for (int i = 0; i < 7; ++i)
        if (dst[i]) PCU(cudaMemcpyAsync(dst[i], p->gcol[i].p, (size_t)n * esz[i], cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaEventRecord(p->ev[1], p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    PCU(cudaEventElapsedTime(&p->ms_d2h, p->ev[0], p->ev[1]));
    return WFL_OK;
}

/* CUDA-event times of the last parse: H2D of the text, kernels, D2H of the columns (milliseconds). */
int wfl_parser_times(const wfl_parser *p, float *ms_h2d, float *ms_kernels, float *ms_d2h) {
    if (!p) return WFL_ERR_ARG;
    if (ms_h2d) *ms_h2d = p->ms_h2d;
    if (ms_kernels) *ms_kernels = p->ms_kernels;
    if (ms_d2h) *ms_d2h = p->ms_d2h;
    return WFL_OK;
}

}  // extern "C"
