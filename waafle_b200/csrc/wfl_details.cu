// --write-details table on the device (write_details, waafle_orgscorer.py:766-812): the text rows
//     contig \t iteration \t clade \t gene_scores \t gene_spans \n
// of every (contig, evaluated level) segment of the exact pipeline's details dump (wfl_pipeline.cu, det_*).
//
// One warp per segment.  It sorts the segment's dump entries by (clade, locus) and drops the duplicates a replayed
// contig leaves, then stages the contig's attached (hit, retained locus) pairs with the hit's clade at that level
// (hit_matches / hit_slice / the ancestor table, shared with the scoring kernels), sorts them by (clade, locus, slice
// start) and merges the slices of every (clade, locus) into the spans of its site array.  A lane writes one row.
// The same code counts (length pass, text == null) and writes (write pass).
#include <algorithm>

#include "wfl_warp_sort.cuh"

namespace wfl {
namespace {

// ---- "{:.3f}" of a double, exactly as Python prints it ----------------------------------------------------------
// x = m * 2^e with an integer mantissa m < 2^53.  For |x| < 2^53, 1000 * m < 2^63 fits a u64, so
// q = round(1000 * x) is computed exactly: (1000 m) >> -e with the remainder compared against one half, ties to even.
// For -e >= 64 the value is below 2^-11 and 1000 m < 2^63 <= 2^(-e-1), so it rounds to 0.  The sign is the sign bit,
// which gives Python's "-0.000" for -0.0 and for negatives that round to zero.  Returns the length, or -1 for
// |x| >= 2^53, infinities and NaN.
__device__ __noinline__ int format3(double x, char *out) {
    const u64 u = (u64)__double_as_longlong(x);
    const bool neg = (u >> 63) != 0;
    const int ex = (int)((u >> 52) & 0x7ff);
    u64 m = u & ((1ull << 52) - 1);
    if (ex == 0x7ff) return -1;
    if (ex) m |= 1ull << 52;
    const int e = (ex ? ex : 1) - 1075;
    u64 q;
    if (e > 0) {
        return -1;   // m >= 2^52 and e >= 1: |x| >= 2^53
    } else if (e == 0) {
        q = m * 1000ull;
    } else if (-e >= 64) {
        q = 0;
    } else {
        const int s = -e;
        const u64 p = m * 1000ull, half = 1ull << (s - 1);
        const u64 r = p & ((1ull << s) - 1);
        q = p >> s;
        if (r > half || (r == half && (q & 1ull))) ++q;
    }
    char tmp[24];
    int n = 0;
    u64 ip = q / 1000ull;
    const int fp = (int)(q % 1000ull);
    tmp[n++] = (char)('0' + fp % 10);
    tmp[n++] = (char)('0' + fp / 10 % 10);
    tmp[n++] = (char)('0' + fp / 100);
    tmp[n++] = '.';
    do { tmp[n++] = (char)('0' + ip % 10); ip /= 10; } while (ip);
    if (neg) tmp[n++] = '-';
    if (out)
        for (int i = 0; i < n; ++i) out[i] = tmp[n - 1 - i];
    return n;
}

// text sink: counts always, writes when p != null
struct Sink {
    char *p;
    long long n;
    __device__ void put(char ch) { if (p) p[n] = ch; ++n; }
    __device__ void str(const char *s, long long len) {
        if (p) for (long long i = 0; i < len; ++i) p[n + i] = s[i];
        n += len;
    }
    __device__ void num(long long v) {
        char t[20];
        int k = 0;
        do { t[k++] = (char)('0' + v % 10); v /= 10; } while (v);
        while (k) put(t[--k]);
    }
};

// scratch bytes of one segment: retained loci, row heads, the two key arrays
__device__ __forceinline__ long long seg_need(int G, int len, int M) {
    return 16ll * (pow2_at_least(len) + pow2_at_least(max(M, 1))) + 4ll * ((G + 3) & ~3) + 4ll * ((len + 3) & ~3) + 64;
}

}  // namespace

__global__ void __launch_bounds__(256) wfl_details_segments_kernel(const DetTextArgs a) {
    const long long n = a.n_dump;
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < n; o += (long long)gridDim.x * blockDim.x) {
        const int c = a.dc[o], it = a.di[o];
        if (o > 0 && a.dc[o - 1] == c && a.di[o - 1] == it) continue;
        long long e = o + 1;
        while (e < n && a.dc[e] == c && a.di[e] == it) ++e;
        const unsigned int s = atomicAdd(a.n_found, 1u);
        DetSeg d;
        d.start = o;
        d.len = (int)(e - o);
        d.contig = c;
        d.iter = it;
        d.pad = 0;
        a.found[s] = d;
    }
}

__global__ void __launch_bounds__(256) wfl_details_rows_kernel(const DetTextArgs a) {
    const int lane = lane_id();
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const DevParams &P = a.P;
    char *slice = a.scratch + warp * a.slice;
    for (long long w = warp; w < a.n_list; w += nwarps) {
        const int si = a.list ? a.list[w] : (int)(a.s0 + w);
        const DetSeg sg = a.seg[si];
        const int c = sg.contig;
        const long long h0 = a.b.hit_off[c], l0 = a.b.locus_off[c];
        const int H = (int)(a.b.hit_off[c + 1] - h0), Graw = (int)(a.b.locus_off[c + 1] - l0);
        // retained loci (attach_loci, waafle_orgscorer.py:350-352) and the attached (hit, locus) pairs
        int G = 0;
#pragma unroll 1
        for (int j = 0; j < Graw; ++j) {
            const int s = a.b.locus_start[l0 + j], e = a.b.locus_end[l0 + j];
            G += (double)(max(s, e) - min(s, e) + 1) >= P.p.min_gene_length;
        }
        int M = 0;
#pragma unroll 1
        for (int base = 0; base < H; base += 32) {
            const int h = base + lane;
            int q1 = 0, q2 = 0;
            const bool hok = h < H && hit_scov_ok(a.b, h0 + h, P.p.min_scov);
            if (h < H) hit_span(a.b, h0 + h, q1, q2);
            const signed char hs = h < H ? hit_strand_of(a.b, h0 + h) : 0;
            int cnt = 0;
#pragma unroll 1
            for (int j = 0; j < Graw && hok; ++j) {
                const int s = a.b.locus_start[l0 + j], e = a.b.locus_end[l0 + j];
                const int lmin = min(s, e), llen = max(s, e) - lmin + 1;
                if ((double)llen >= P.p.min_gene_length &&
                    hit_matches(P, min(q1, q2), max(q1, q2), hs, lmin, llen, a.b.locus_strand[l0 + j]))
                    ++cnt;
            }
            M += warp_sum(cnt);
        }
        const long long need = seg_need(G, sg.len, M);
        if (need > a.slice) {   // handed to a second launch with larger slices
            if (lane == 0) {
                a.defer[atomicAdd(a.n_defer, 1u)] = si;
                atomicMax(a.max_need, (unsigned long long)need);
            }
            continue;
        }
        const int NE = pow2_at_least(sg.len), NA = pow2_at_least(max(M, 1));
        ulonglong2 *ent = reinterpret_cast<ulonglong2 *>(slice);
        ulonglong2 *att = ent + NE;
        int *kept = reinterpret_cast<int *>(att + NA);
        int *rowh = kept + ((G + 3) & ~3);
        // dump entries: key (clade, raw locus), payload the entry index
        for (int i = lane; i < NE; i += 32) {
            ulonglong2 k = make_ulonglong2(~0ull, ~0ull);
            if (i < sg.len) {
                const long long o = sg.start + i;
                k.x = ((u64)(u32)a.dc_clade[o] << 32) | (u32)a.dl[o];
                k.y = (u64)o;
            }
            ent[i] = k;
        }
        if (lane == 0) {
            int g = 0;
            for (int j = 0; j < Graw; ++j) {
                const int s = a.b.locus_start[l0 + j], e = a.b.locus_end[l0 + j];
                if ((double)(max(s, e) - min(s, e) + 1) >= P.p.min_gene_length) kept[g++] = j;
            }
        }
        // attached pairs at this level: key (clade, retained locus k), (slice start, slice end)
        const int row = min(P.p.jump_taxonomy + sg.iter, a.anc_rows - 1);
        const int *anc = a.anc + (size_t)row * (size_t)a.t.n_nodes;
        int fill = 0;
#pragma unroll 1
        for (int base = 0; base < H; base += 32) {
            const int h = base + lane;
            int q1 = 0, q2 = 0, cl = 0;
            const bool hok = h < H && hit_scov_ok(a.b, h0 + h, P.p.min_scov);
            double sc = 0.0;
            if (h < H) {
                hit_span(a.b, h0 + h, q1, q2);
                int tx = hit_taxon_of(a.b, h0 + h);
                if ((u32)tx >= (u32)a.t.n_nodes) tx = a.t.root;
                cl = anc[tx];
                sc = a.b.hit_score[h0 + h];
            }
            const signed char hs = h < H ? hit_strand_of(a.b, h0 + h) : 0;
            const int hmin = min(q1, q2), hmax = max(q1, q2);
            int k = 0;
#pragma unroll 1
            for (int j = 0; j < Graw; ++j) {
                const int s = a.b.locus_start[l0 + j], e = a.b.locus_end[l0 + j];
                const int lmin = min(s, e), llen = max(s, e) - lmin + 1;
                if (!((double)llen >= P.p.min_gene_length)) continue;
                const bool mt = hok && hit_matches(P, hmin, hmax, hs, lmin, llen, a.b.locus_strand[l0 + j]);
                const u32 m = __ballot_sync(FULL, mt);
                if (mt) {
                    int s1, e1;
                    hit_slice(hmin, hmax, lmin, llen, s1, e1);
                    if (!(sc > 0.0)) e1 = s1;   // the site array exists but this hit leaves it at zero
                    att[fill + __popc(m & lt_mask())] = make_ulonglong2(((u64)(u32)cl << 32) | (u32)k, ((u64)(u32)s1 << 32) | (u32)e1);
                }
                fill += __popc(m);
                ++k;
            }
        }
        for (int i = M + lane; i < NA; i += 32) att[i] = make_ulonglong2(~0ull, ~0ull);
        __syncwarp();
        warp_sort(ent, NE);
        warp_sort(att, NA);
        // row heads: the first entry of every clade; entries equal to their predecessor (a replay) are skipped below
        int nrows = 0;
#pragma unroll 1
        for (int base = 0; base < sg.len; base += 32) {
            const int i = base + lane;
            const bool head = i < sg.len && (i == 0 || (ent[i].x >> 32) != (ent[i - 1].x >> 32));
            const u32 m = __ballot_sync(FULL, head);
            if (head) rowh[nrows + __popc(m & lt_mask())] = i;
            nrows += __popc(m);
        }
        __syncwarp();
        long long seg_base = a.text ? a.text_off[si] - a.text_base : 0, seg_bytes = 0;
        const char *cname = a.cname + a.cname_off[c];
        const long long cname_len = a.cname_off[c + 1] - a.cname_off[c];
#pragma unroll 1
        for (int base = 0; base < nrows; base += 32) {
            const int r = base + lane;
            long long len = 0;
            // two rounds with a text buffer (count, then write at the scanned offset), one without
#pragma unroll 1
            for (int round = 0; round < (a.text ? 2 : 1); ++round) {
                long long off = 0;
                if (round == 1) {
                    long long inc = len;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const long long t = __shfl_up_sync(FULL, inc, o);
                        if (lane >= o) inc += t;
                    }
                    off = inc - len;
                }
                if (r < nrows) {
                    const int rs = rowh[r], re = r + 1 < nrows ? rowh[r + 1] : sg.len;
                    const u32 clade = (u32)(ent[rs].x >> 32);
                    Sink o{round ? a.text + seg_base + seg_bytes + off : nullptr, 0};
                    o.str(cname, cname_len);
                    o.put('\t');
                    o.num(max(1, sg.iter));   // ITERATION: 1, 1, 2, 3, ... (OS:566-579)
                    o.put('\t');
                    o.str(a.tname + a.tname_off[clade], a.tname_off[clade + 1] - a.tname_off[clade]);
                    o.put('\t');
                    int p = rs;
#pragma unroll 1
                    for (int k = 0; k < G; ++k) {
                        if (k) o.put('|');
                        while (p < re && (int)(u32)ent[p].x < kept[k]) ++p;
                        if (p < re && (int)(u32)ent[p].x == kept[k]) {
                            const int n = format3(a.ds[ent[p].y], o.p ? o.p + o.n : nullptr);
                            if (n < 0) { atomicAdd(a.err, 1u); break; }
                            o.n += n;
                        } else {
                            o.str("0.000", 5);   // no group of this clade on the locus (:404-405)
                        }
                    }
                    o.put('\t');
                    // gene spans (make_gene_spans_field, :773-791): the clade's attached pairs, grouped by locus
                    int lo = 0, hi = M;
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        if ((u32)(att[mid].x >> 32) < clade) lo = mid + 1; else hi = mid;
                    }
                    const long long field0 = o.n;
                    int q = lo;
#pragma unroll 1
                    for (int k = 0; k < G; ++k) {
                        if (k) o.put('|');
                        if (!(q < M && att[q].x == (((u64)clade << 32) | (u32)k))) {
                            o.str("None", 4);   // no site array for this clade / locus (:776-781)
                            continue;
                        }
                        int ca = -1, cb = -1;
                        bool first = true;
                        for (; q < M && att[q].x == (((u64)clade << 32) | (u32)k); ++q) {
                            const int sa = (int)(att[q].y >> 32), sb = (int)(u32)att[q].y;
                            if (sb <= sa) continue;
                            if (ca >= 0 && sa <= cb) { cb = max(cb, sb); continue; }
                            if (ca >= 0 && cb - ca >= 2) {
                                if (!first) o.put(':');
                                o.num(ca + 1); o.put(':'); o.num(cb);
                                first = false;
                            }
                            ca = sa;
                            cb = sb;
                        }
                        if (ca >= 0 && cb - ca >= 2) {
                            if (!first) o.put(':');
                            o.num(ca + 1); o.put(':'); o.num(cb);
                        }
                    }
                    if (o.n == field0) o.str("--", 2);   // an empty field (format_field, utils.py:137-139)
                    o.put('\n');
                    len = o.n;
                }
            }
            long long tot = len;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(FULL, tot, o);
            seg_bytes += tot;
        }
        if (lane == 0 && !a.text) a.seg_bytes[si] = seg_bytes;
        __syncwarp();
    }
}

__global__ void wfl_format3_kernel(const double *x, long long n, char *text, int *len, unsigned int *err) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int k = format3(x[i], text + 24 * i);
        len[i] = k;
        if (k < 0) atomicAdd(err, 1u);
    }
}

void launch_details_segments(const DetTextArgs &a, cudaStream_t s) {
    const long long blocks = std::min<long long>((a.n_dump + 255) / 256, 4096);
    wfl_details_segments_kernel<<<(int)std::max<long long>(1, blocks), 256, 0, s>>>(a);
}

void launch_details_rows(const DetTextArgs &a, long long warps, cudaStream_t s) {
    wfl_details_rows_kernel<<<(int)std::max<long long>(1, (warps + 7) / 8), 256, 0, s>>>(a);
}

void launch_format3(const double *x, long long n, char *text, int *len, unsigned int *err, cudaStream_t s) {
    const long long blocks = std::min<long long>((n + 255) / 256, 4096);
    wfl_format3_kernel<<<(int)std::max<long long>(1, blocks), 256, 0, s>>>(x, n, text, len, err);
}

}  // namespace wfl
