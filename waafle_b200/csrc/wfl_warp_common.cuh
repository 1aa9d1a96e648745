// Warp-synchronous device helpers shared by the warp-per-contig kernels (wfl_pipeline.cu: the exact path as
// instruction-cache-sized phase kernels; wfl_fast.cu: the fused shared-memory fast path, which calls the exact
// K2 code below for gene scores that land inside its guard band).
#pragma once

#include "wfl_device.cuh"

namespace wfl {
namespace {

typedef unsigned long long u64;
typedef unsigned int u32;
typedef unsigned short u16;
typedef unsigned char u8;

constexpr u32 FULL = 0xffffffffu;
constexpr int MAXDEPTH = 28;   // pairwise tree depth for n < 2^31
constexpr int BITMAP_MAX_WORDS = 1024;   // taxonomies up to 32768 nodes use the bitmap clade table
#ifndef WFL_K2_TWO
#define WFL_K2_TWO 1     // closed form for leaves with two run boundaries
#endif
constexpr int RMAX = 6;        // envelope runs handled per mixed leaf before the per-site fallback

// Order-preserving map double -> u64 (max on the bits == max on the doubles).
__device__ __forceinline__ u64 dbits(double x) {
    if (x == 0.0) x = 0.0;   // -0.0 -> +0.0
    u64 u = (u64)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double dbits_inv(u64 b) {
    u64 u = (b >> 63) ? (b & 0x7fffffffffffffffull) : ~b;
    return __longlong_as_double((long long)u);
}

struct Arena {
    char *smem, *slab;
    size_t smem_cap, slab_cap, smem_used, slab_used;
    bool ok, all_smem;
    __device__ __noinline__ void *raw(size_t bytes) {
        bytes = (bytes + 15) & ~size_t(15);
        if (smem_used + bytes <= smem_cap) {
            void *p = smem + smem_used;
            smem_used += bytes;
            return p;
        }
        all_smem = false;
        if (slab_used + bytes <= slab_cap) {
            void *p = slab + slab_used;
            slab_used += bytes;
            return p;
        }
        ok = false;
        return nullptr;
    }
    template <class T>
    __device__ __forceinline__ T *get(size_t n) { return static_cast<T *>(raw(n * sizeof(T))); }
};

// ---- hit columns in either wire format (wide wfl_batch / compact wfl_packed_batch) -----------------
__device__ __forceinline__ void hit_span(const DevBatch &b, long long h, int &q1, int &q2) {
    if (b.hit_tax16) { q1 = b.hit_qstart16[h]; q2 = b.hit_qend16[h]; }
    else { q1 = b.hit_qstart[h]; q2 = b.hit_qend[h]; }
}
// scov_modified >= --min-scov (waafle_orgscorer.py:362); the compact format carries the host's verdict in bit 15
__device__ __forceinline__ bool hit_scov_ok(const DevBatch &b, long long h, double min_scov) {
    return b.hit_tax16 ? (b.hit_tax16[h] & 0x8000u) != 0u : b.hit_scov[h] >= min_scov;
}
__device__ __forceinline__ signed char hit_strand_of(const DevBatch &b, long long h) {
    return b.hit_tax16 ? ((b.hit_tax16[h] & 0x4000u) ? '-' : '+') : b.hit_strand[h];
}
__device__ __forceinline__ int hit_taxon_of(const DevBatch &b, long long h) {
    return b.hit_tax16 ? (int)(b.hit_tax16[h] & 0x3fffu) : b.hit_taxon[h];
}
__device__ __forceinline__ u32 hit_sysmask_of(const DevBatch &b, long long h) {
    return b.hit_tax16 ? (u32)b.hit_sysmask8[h] : b.hit_sysmask[h];
}

// ---- warp primitives -----------------------------------------------------------------------
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ u32 lt_mask() { return (1u << lane_id()) - 1u; }

__device__ __noinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __noinline__ u64 warp_max_u64(u64 v) {
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) {
        u64 t = __shfl_xor_sync(FULL, v, o);
        v = t > v ? t : v;
    }
    return v;
}
__device__ __noinline__ long long warp_max_ll(long long v) {
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) {
        long long t = __shfl_xor_sync(FULL, v, o);
        v = t > v ? t : v;
    }
    return v;
}
__device__ __noinline__ int warp_excl_scan(int v, int &total) {
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(FULL, inc, o);
        if (lane_id() >= o) inc += t;
    }
    total = __shfl_sync(FULL, inc, 31);
    return inc - v;
}

// LCA by depth-aligned parent walk == deepest common prefix of root-first lineages
// (waafle/utils.py:401-411).  -1 is the identity.
__device__ __noinline__ int lca2(const DevTax &t, int a, int b) {
    if (a < 0) return b;
    if (b < 0) return a;
    int da = t.depth[a], db = t.depth[b];
#pragma unroll 1
    while (da > db) { a = t.parent[a]; --da; }
#pragma unroll 1
    while (db > da) { b = t.parent[b]; --db; }
#pragma unroll 1
    while (a != b) { a = t.parent[a]; b = t.parent[b]; }
    return a;
}
__device__ __noinline__ int warp_lca(const DevTax &t, int v) {
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) v = lca2(t, v, __shfl_xor_sync(FULL, v, o));
    return v;
}

// Stable warp multisplit of the item sequence src[0..n) (identity if src == nullptr) by bin key[item]
// in [0, nbins): out[] receives the items grouped by bin, sequence order kept inside each bin.  `cur` is an nbins+1 scratch array;
// on return cur[b] = end of bin b (== start of bin b+1).
__device__ __noinline__ void warp_multisplit(int n, int nbins, const int *key, const int *src, int *cur, int *out) {
    const int lane = lane_id();
#pragma unroll 1
    for (int b = lane; b <= nbins; b += 32) cur[b] = 0;
    __syncwarp();
#pragma unroll 1
    for (int base = 0; base < n; base += 32) {
        int i = base + lane;
        int b = i < n ? key[src ? src[i] : i] : nbins;
        u32 peers = __match_any_sync(FULL, b);
        if ((peers & lt_mask()) == 0) cur[b] += __popc(peers);
        __syncwarp();
    }
    int carry = 0;
#pragma unroll 1
    for (int base = 0; base < nbins; base += 32) {
        int b = base + lane, c = b < nbins ? cur[b] : 0, tot;
        int ex = warp_excl_scan(c, tot);
        if (b < nbins) cur[b] = carry + ex;
        carry += tot;
    }
    __syncwarp();
#pragma unroll 1
    for (int base = 0; base < n; base += 32) {
        int i = base + lane;
        int it = i < n ? (src ? src[i] : i) : 0;
        int b = i < n ? key[it] : nbins;
        u32 peers = __match_any_sync(FULL, b);
        if (i < n) out[cur[b] + __popc(peers & lt_mask())] = it;
        __syncwarp();
        if (i < n && (peers & lt_mask()) == 0) cur[b] += __popc(peers);
        __syncwarp();
    }
}

// ---- numpy pairwise summation ---------------------------------------------------------------
// numpy/_core/src/umath/loops_utils.h.src DOUBLE_pairwise_sum: n < 8 plain loop; n <= 128 eight
// strided accumulators r[j] += a[i+j], res = ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the n%8
// tail; otherwise split at n2 = n/2 - (n/2)%8 and add the two halves.
//
// The split tree depends only on n, so it is flattened once per locus into a leaf plan shared by
// all clades: plan entry = leaf size m | (#pending left sums to add after this leaf) << 8.

// K2-HOST-BEGIN (tests/test_k2_host.py compiles everything up to K2-HOST-END for the host)
// Emit the leaf plan of an n-element sum (at most plan_cap(n) entries).  Every leaf of a split
// node has more than 56 elements, hence the bound.
__device__ __forceinline__ int plan_cap(int n) { return n / 57 + 2; }

__device__ __noinline__ int build_plan(int n, u16 *plan, u8 *k8set) {
    int sz[MAXDEPTH], ch[MAXDEPTH], sp = 0, cnt = 0, nset = 0;
    sz[0] = n;
    ch[0] = 0;
    sp = 1;
    while (sp > 0) {
        int m = sz[--sp], c = ch[sp];
        if (m <= 128) {
            if (plan) {
                plan[cnt] = (u16)(m | (c << 8));
                if (m >= 8 && nset <= 4) {   // distinct lane counts m/8, ascending, for the S_k memo
                    u8 k = (u8)(m >> 3);
                    int j = 0;
                    while (j < nset && k8set[j] < k) ++j;
                    if (j == nset || k8set[j] != k) {
                        if (nset < 4) {
#pragma unroll 1
                            for (int q = nset; q > j; --q) k8set[q] = k8set[q - 1];
                            k8set[j] = k;
                        }
                        ++nset;
                    }
                }
            }
            ++cnt;
        } else {
            int n2 = m / 2;
            n2 -= n2 % 8;
            sz[sp] = m - n2;   // right half: evaluated second, then added to the pending left sum
            ch[sp++] = c + 1;
            sz[sp] = n2;
            ch[sp++] = 0;
        }
    }
    if (plan) {
#pragma unroll 1
        for (int q = nset < 4 ? nset : 4; q < 4; ++q) k8set[q] = 0;
        if (nset > 4) k8set[0] = k8set[1] = k8set[2] = k8set[3] = 0;   // too many sizes: no memo
    }
    return cnt;
}

// Envelope run starting at `pos` for one (clade, locus) group whose records are ra/rb/rv[rs..re)
// (copies in group order): returns its end, *v its value.
__device__ __noinline__ int site_advance(const int *ra, const int *rb, const double *rv, int rs, int re, int n,
                                         bool sorted, int pos, double *vout) {
    double v = 0.0;   // np.zeros(len(locus)), waafle_orgscorer.py:381
    int nx = n;
#pragma unroll 1
    for (int r = rs; r < re; ++r) {
        int a = ra[r], b = rb[r];
        if (a <= pos && pos < b) {
            v = fmax(v, rv[r]);   // np.maximum(slice, score), waafle_orgscorer.py:382
            nx = min(nx, b);
            if (sorted) break;    // descending score order: the first cover is the max
        } else if (a > pos) {
            nx = min(nx, a);
        }
    }
    *vout = v;
    return nx;
}

// One (clade, locus) group: envelope of its records streamed as constant runs.
struct Site {
    const int *ra, *rb;   // python-slice [a, b) of the group's records, [rs..re) in group order
    const double *rv;     // their waafle_scores
    int rs, re, n;
    bool sorted;          // records in descending score order -> first covering record is the max
    int pos, run_end;
    double run_v;
    // memo of the add chains S_k(v) = v+v+...+v (k terms, sequential) for the current run
    double Sk[4];
    u8 k8[4];
    bool memo_ok;

    __device__ __forceinline__ void advance() {
        run_end = site_advance(ra, rb, rv, rs, re, n, sorted, pos, &run_v);
        memo_ok = false;
    }
    __device__ __forceinline__ double next() {
        if (pos >= run_end) advance();
        ++pos;
        return run_v;
    }
    // S_k(run_v) for k = m/8 lanes
    __device__ __forceinline__ double chain(int k) {
        const double v = run_v;
        if (k8[0]) {
            if (!memo_ok) {
                double r = v;
                int i = 1;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    int kk = k8[j];
#pragma unroll 1
                    for (; i < kk; ++i) r += v;
                    Sk[j] = r;
                }
                memo_ok = true;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (k8[j] == k) return Sk[j];
        }
        double r = v;
#pragma unroll 1
        for (int i = 1; i < k; ++i) r += v;
        return r;
    }
};

// A leaf that lies inside one run.
__device__ __forceinline__ double const_leaf(Site &s, int m) {
    const double v = s.run_v;
    s.pos += m;
    if (v == 0.0) return 0.0;
    double res;
    if (m < 8) {
        res = 0.0;
#pragma unroll 1
        for (int i = 0; i < m; ++i) res += v;
        return res;
    }
    res = 8.0 * s.chain(m >> 3);   // ((r+r)+(r+r))+((r+r)+(r+r)) with eight equal lanes: exact
#pragma unroll 1
    for (int i = 0; i < (m & 7); ++i) res += v;
    return res;
}

// COLD path, kept out of line so that the hot leaf code stays compact in the instruction cache: a leaf of
// a gene shorter than 8 sites, or a leaf with more than RMAX runs -- literal per-site evaluation.
__device__ __noinline__ double literal_leaf(const int *ra, const int *rb, const double *rv, int rs, int re, int n,
                                            bool sorted, int p0, int m) {
    Site s;
    s.ra = ra; s.rb = rb; s.rv = rv;
    s.rs = rs; s.re = re; s.n = n; s.sorted = sorted;
    s.k8[0] = s.k8[1] = s.k8[2] = s.k8[3] = 0;
    s.memo_ok = false;
    s.pos = p0;
    s.run_end = p0;
    s.run_v = 0.0;
    if (m < 8) {
        double r = 0.0;
#pragma unroll 1
        for (int i = 0; i < m; ++i) r += s.next();
        return r;
    }
    const int k8 = m >> 3, body = k8 << 3;
    double r[8];
#pragma unroll 1
    for (int j = 0; j < 8; ++j) r[j] = s.next();
#pragma unroll 1
    for (int c = 1; c < k8; ++c) {
#pragma unroll 1
        for (int j = 0; j < 8; ++j) r[j] += s.next();
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll 1
    for (int p = body; p < m; ++p) res += s.next();
    return res;
}

// A leaf that contains envelope breakpoints.
__device__ __forceinline__ double mixed_leaf(Site &s, int m) {
    const int p0 = s.pos;
    if (m < 8) {
        const double r = literal_leaf(s.ra, s.rb, s.rv, s.rs, s.re, s.n, s.sorted, p0, m);
        s.pos = s.run_end = p0 + m;   // the next leaf re-reads its run
        return r;
    }
    // collect the runs that intersect the leaf (ends relative to the leaf start)
    int rend[RMAX];
    double rval[RMAX];
    int nr = 0;
    u32 brk = 0;   // (boundary & 7) of the interior run boundaries
#pragma unroll 1
    for (;;) {
        if (s.pos >= s.run_end) s.advance();
        int e = min(s.run_end - p0, m);
        if (nr == RMAX) { nr = -1; break; }
        rend[nr] = e;
        rval[nr] = s.run_v;
        ++nr;
        if (e >= m) break;
        brk |= 1u << (e & 7);
        s.pos = p0 + e;
    }
    const int k8 = m >> 3, body = k8 << 3;
    if (nr == 2 && rend[0] < body) {
        // The common case: ONE run boundary b inside the leaf body, v0 before it and v1 after it.
        // With b = 8*c0 + j0, columns j < j0 hold c0+1 copies of v0 then k8-c0-1 copies of v1 and
        // columns j >= j0 hold c0 copies of v0 then k8-c0 copies of v1: two add chains that share
        // their v0 prefix.  (One of v0 / v1 is usually 0 -- the flank of a hit -- and adds nothing.)
        const int b = rend[0], c0 = b >> 3, j0 = b & 7;
        const double v0 = rval[0], v1 = rval[1];
        double x, y;   // column sums of the two classes
        if (c0 == 0) {
            x = v0;    // one copy of v0 ...
            y = v1;    // ... or none: the column starts with v1
            if (v1 != 0.0) {
#pragma unroll 1
                for (int i = 1; i < k8; ++i) { x += v1; y += v1; }
            }
        } else {
            y = v0;
            if (v0 != 0.0) {
#pragma unroll 1
                for (int i = 1; i < c0; ++i) y += v0;   // S_c0(v0)
            }
            x = y + v0;                                 // S_{c0+1}(v0)
            if (v1 != 0.0) {
                const int nx = k8 - c0 - 1;
#pragma unroll 1
                for (int i = 0; i < nx; ++i) { x += v1; y += v1; }
                y += v1;                                // the lower class holds one more v1
            }
        }
        // fold ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) with r_j = (j < j0 ? x : y)
        const double r0 = 0 < j0 ? x : y, r1 = 1 < j0 ? x : y, r2 = 2 < j0 ? x : y, r3 = 3 < j0 ? x : y;
        const double r4 = 4 < j0 ? x : y, r5 = 5 < j0 ? x : y, r6 = 6 < j0 ? x : y;
        double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + y));
#pragma unroll 1
        for (int p = body; p < m; ++p) res += v1;   // the n % 8 tail lies behind the boundary
        s.pos = p0 + m;
        return res;
    }
#if WFL_K2_TWO
    if (nr == 3 && rend[0] < body) {
        // TWO boundaries b1 < b2 (typically a lower-scoring hit sticking out of the best one next to the
        // zero flank): column j holds n0(j) copies of v0, then v1 up to n01(j), then v2, with
        // n0(j) = (b1 >> 3) + (j < (b1 & 7)) and n01(j) = min(k8, (b2 >> 3) + (j < (b2 & 7))) -- at most three
        // distinct columns, split at t1 <= t2.  All state in registers.
        const int b1 = rend[0], b2 = rend[1];
        const double v0 = rval[0], v1 = rval[1], v2 = rval[2];
        const int J1 = b1 & 7, J2 = (b2 >> 3) < k8 ? (b2 & 7) : 0;
        const int t1 = min(J1, J2), t2 = max(J1, J2);
        double xa = 0.0, xb = 0.0, xc = 0.0;
#pragma unroll 1
        for (int q = 0; q < 3; ++q) {
            const int j = q == 0 ? 0 : (q == 1 ? t1 : t2);
            if ((q == 0 && t1 == 0) || (q == 1 && t2 == t1)) continue;   // empty class
            const int n0 = (b1 >> 3) + (j < J1), n01 = min(k8, (b2 >> 3) + (j < (b2 & 7)));
            double acc = 0.0;   // 0 + v == v: the first term needs no special case
            if (v0 != 0.0) {
#pragma unroll 1
                for (int i = 0; i < n0; ++i) acc += v0;
            }
            if (v1 != 0.0) {
#pragma unroll 1
                for (int i = n0; i < n01; ++i) acc += v1;
            }
            if (v2 != 0.0) {
#pragma unroll 1
                for (int i = n01; i < k8; ++i) acc += v2;
            }
            if (q == 0) xa = acc; else if (q == 1) xb = acc; else xc = acc;
        }
        const double r0 = 0 < t1 ? xa : (0 < t2 ? xb : xc), r1 = 1 < t1 ? xa : (1 < t2 ? xb : xc);
        const double r2 = 2 < t1 ? xa : (2 < t2 ? xb : xc), r3 = 3 < t1 ? xa : (3 < t2 ? xb : xc);
        const double r4 = 4 < t1 ? xa : (4 < t2 ? xb : xc), r5 = 5 < t1 ? xa : (5 < t2 ? xb : xc);
        const double r6 = 6 < t1 ? xa : (6 < t2 ? xb : xc);
        double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + xc));
#pragma unroll 1
        for (int p = body; p < m; ++p) res += p < b2 ? v1 : v2;   // the n % 8 tail lies behind b1
        s.pos = p0 + m;
        return res;
    }
#endif
    if (nr > 0) {
        // column j accumulates a[j], a[8+j], ...: runs enter it as (count, value) stretches;
        // neighbouring columns differ only where a run boundary b has b % 8 == j.  The eight
        // column sums are folded into ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) as they appear.
        double acc = 0.0, pair = 0.0, quad = 0.0, half = 0.0, res = 0.0;
#pragma unroll 1
        for (int j = 0; j < 8; ++j) {
            if (j == 0 || ((brk >> j) & 1)) {
                acc = 0.0;
                bool first = true;
                int start = 0;
#pragma unroll 1
                for (int q = 0; q < nr; ++q) {
                    int e = min(rend[q], body);
                    int c_lo = start <= j ? 0 : (start - j + 7) >> 3;
                    int c_hi = e <= j ? 0 : (e - j + 7) >> 3;
                    int cnt = c_hi - c_lo;
                    start = rend[q];
                    if (cnt <= 0) continue;
                    const double v = rval[q];
                    if (first) {
                        acc = v;
                        --cnt;
                        first = false;
                    }
                    if (v != 0.0) {
#pragma unroll 1
                        for (int i = 0; i < cnt; ++i) acc += v;
                    }
                }
            }
            if ((j & 1) == 0) {
                pair = acc;
            } else {
                pair = pair + acc;                       // r[j-1] + r[j]
                if ((j & 2) == 0) {
                    quad = pair;
                } else {
                    quad = quad + pair;                  // (r[j-3]+r[j-2]) + (r[j-1]+r[j])
                    if (j == 3) half = quad; else res = half + quad;
                }
            }
        }
        int q = 0;
#pragma unroll 1
        for (int p = body; p < m; ++p) {   // the n % 8 tail of the last leaf
            while (rend[q] <= p) ++q;
            res += rval[q];
        }
        s.pos = p0 + m;
        return res;
    }
    // more than RMAX runs in one leaf: literal per-site evaluation
    const double res = literal_leaf(s.ra, s.rb, s.rv, s.rs, s.re, s.n, s.sorted, p0, m);
    s.pos = s.run_end = p0 + m;   // the next leaf re-reads its run
    return res;
}

// np.mean of the group's site array (waafle_orgscorer.py:403) without materialising it.
// ra/rb/rv[rs..re) are the group's records (in descending score order if `sorted`).
__device__ __noinline__ double group_mean(const int *ra, const int *rb, const double *rv, int rs, int re, int n,
                                          bool sorted, u32 k8pack, const u16 *plan, int nleaf) {
    Site s;
    s.ra = ra; s.rb = rb; s.rv = rv;
    s.rs = rs; s.re = re; s.n = n; s.sorted = sorted;
    s.k8[0] = (u8)k8pack; s.k8[1] = (u8)(k8pack >> 8); s.k8[2] = (u8)(k8pack >> 16); s.k8[3] = (u8)(k8pack >> 24);
    s.pos = 0;
    s.run_end = 0;
    s.memo_ok = false;
    double st[MAXDEPTH];
    int sp = 0;
#pragma unroll 1
    for (int l = 0; l < nleaf; ++l) {
        const int e = plan[l], m = e & 0xff, nadd = e >> 8;
        if (s.pos >= s.run_end) s.advance();
        double val = (s.run_end - s.pos >= m) ? const_leaf(s, m) : mixed_leaf(s, m);
#pragma unroll 1
        for (int q = 0; q < nadd; ++q) val = st[--sp] + val;
        st[sp++] = val;
    }
    return st[0] / (double)n;
}

// ---- closed-form envelope integral (fast path, wfl_fast.cu) ----
// The records of a group live in a per-locus buffer: bv[r] score (>= 0), bab[r] python slice a | b << 16, visited through
// the order array bord[rs..re).
// Generic envelope integral of one group (records q in [rs, re) of the locus buffer, via bord): sweep over the
// distinct endpoints.  Cold: only groups whose better hits leave a gap.
__device__ __noinline__ double group_integral_general(const double *bv, const u32 *bab, const u16 *bord, int rs, int re) {
    double sum = 0.0;
#pragma unroll 1
    for (int e2 = 2 * rs; e2 < 2 * re; ++e2) {
        const u32 abq = bab[bord[e2 >> 1]];
        const int e = (e2 & 1) ? (int)(abq >> 16) : (int)(abq & 0xffffu);
        bool dup = false;
        int nx = 0x7fffffff;
        double mx = 0.0;
#pragma unroll 1
        for (int q = rs; q < re; ++q) {
            const int r = bord[q];
            const u32 ab = bab[r];
            const int a = (int)(ab & 0xffffu), b = (int)(ab >> 16);
            if (a <= e && e < b) mx = fmax(mx, bv[r]);
            if (a > e) nx = min(nx, a);
            if (b > e) nx = min(nx, b);
            dup |= (a == e && 2 * q < e2) || (b == e && 2 * q + 1 < e2);
        }
        if (!dup && mx > 0.0 && nx != 0x7fffffff) sum += mx * (double)(nx - e);
    }
    return sum;
}

// Closed-form envelope integral of a group with >= 2 records that arrive in DESCENDING SCORE order (the fast path sorts
// every locus' records once per contig; stable splits keep the order inside each group): the union of the records seen
// so far is kept as ONE interval [ua, ub) and every record adds v * (newly covered sites).  A record that leaves a gap
// sends the group to the generic sweep.  n = gene length: once the union covers the gene nothing can be added.
__device__ __forceinline__ double group_integral(const double *bv, const u32 *bab, const u16 *bord, int rs, int re, int n) {
    int r = bord[rs];
    u32 ab = bab[r];
    int ua = (int)(ab & 0xffffu), ub = (int)(ab >> 16);
    double sum = bv[r] * (double)(ub - ua);
#pragma unroll 1
    for (int q = rs + 1; q < re; ++q) {
        if (ua == 0 && ub == n) break;
        r = bord[q];
        const double v = bv[r];
        if (!(v > 0.0)) break;   // descending: the rest contributes nothing
        ab = bab[r];
        const int a = (int)(ab & 0xffffu), b = (int)(ab >> 16);
        if (a > ub || b < ua) return group_integral_general(bv, bab, bord, rs, re);
        const int add = max(0, ua - a) + max(0, b - ub);
        if (add) {
            sum += v * (double)add;
            ua = min(ua, a);
            ub = max(ub, b);
        }
    }
    return sum;
}
// K2-HOST-END

// Generic sequential pairwise sum for the short gene-level vectors of Contig.score.
template <class Src>
__device__ double pw_leaf_seq(Src &s, int m) {
    if (m < 8) {
        double r = 0.0;
#pragma unroll 1
        for (int i = 0; i < m; ++i) r += s.next();
        return r;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = s.next();
#pragma unroll 1
    for (int c = 1; c < (m >> 3); ++c) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] += s.next();
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll 1
    for (int i = 0; i < (m & 7); ++i) res += s.next();
    return res;
}
template <class Src>
__device__ double pairwise_seq(Src &s, int n) {
    if (n <= 128) return pw_leaf_seq(s, n);
    // explicit post-order walk of the split tree (only contigs with > 128 non-ignored loci get here)
    int sz[MAXDEPTH];
    double acc[MAXDEPTH];
    u8 st[MAXDEPTH];
    int sp = 0;
    sz[0] = n;
    st[0] = 0;
    double ret = 0.0;
    bool returning = false;
#pragma unroll 1
    for (;;) {
        if (!returning) {
            int m = sz[sp];
            if (m <= 128) {
                ret = pw_leaf_seq(s, m);
                returning = true;
                if (--sp < 0) break;
            } else {
                int n2 = m / 2;
                n2 -= n2 % 8;
                st[sp] = 1;
                sz[sp + 1] = n2;
                st[++sp] = 0;
            }
        } else if (st[sp] == 1) {
            acc[sp] = ret;
            int m = sz[sp], n2 = m / 2;
            n2 -= n2 % 8;
            st[sp] = 2;
            sz[sp + 1] = m - n2;
            st[++sp] = 0;
            returning = false;
        } else {
            ret = acc[sp] + ret;
            if (--sp < 0) break;
        }
    }
    return ret;
}

// Gene-score rows are sparse: groups sorted by (clade, locus); a missing locus scores 0
// (waafle_orgscorer.py:404-405).
struct RowCursor {
    const int *g_loc;
    const double *g_score;
    int p, e;
    __device__ __forceinline__ double at(int locus) {
        while (p < e && g_loc[p] < locus) ++p;
        return (p < e && g_loc[p] == locus) ? g_score[p] : 0.0;
    }
};
// Values of Contig.score (waafle_orgscorer.py:447-461): max(s1, s2) at the non-ignored loci.
struct ScoreSrc {
    RowCursor r1, r2;
    const u8 *ign;
    int i;
    bool two;
    double crit;
    __device__ __noinline__ double next() {
        while (ign[i]) ++i;
        double v = r1.at(i);
        if (two) v = fmax(v, r2.at(i));
        ++i;
        crit = fmin(crit, v);
        return v;
    }
};

struct Level {   // per-level views shared by the search routines (all pointers arena-backed)
    int G, W, T, Ngrp, n_unmasked;
    const int *g_loc;
    const double *g_score;
    const int *cl_id, *cl_go;
    const u64 *mk[3];   // per clade gene bitmasks: score >= k1 / k2 / c_eps
    const u64 *um;      // non-ignored loci
    const u8 *ign;
    const int *l_len;
    const int *cl_par;   // parent of each listed clade (get_sisters works on the taxonomy file's rows), else -1
};

__device__ __noinline__ double score_clades(const Level *L, int t1, int t2, double *crit_out) {
    ScoreSrc s;
    s.r1 = RowCursor{L->g_loc, L->g_score, L->cl_go[t1], L->cl_go[t1 + 1]};
    s.two = t2 >= 0;
    s.r2 = s.two ? RowCursor{L->g_loc, L->g_score, L->cl_go[t2], L->cl_go[t2 + 1]} : s.r1;
    s.ign = L->ign;
    s.i = 0;
    s.crit = __longlong_as_double(0x7ff0000000000000ll);
    const int n = L->n_unmasked;
    double sum = pairwise_seq(s, n);
    *crit_out = s.crit;
    return sum / (double)n;   // np.mean = add.reduce / n
}

// Letters of a two-clade option on word w (waafle_orgscorer.py:524-534), before the A/B swap.
__device__ __forceinline__ void letters(const Level &L, const u64 *mamb, bool unknown_involved, int t1,
                                        int t2, int w, u64 &A, u64 &B, u64 &amb) {
    u64 um = L.um[w];
    amb = unknown_involved ? 0ull : (mamb[(size_t)t1 * L.W + w] & mamb[(size_t)t2 * L.W + w] & um);
    A = L.mk[1][(size_t)t1 * L.W + w] & um & ~amb;
    B = L.mk[1][(size_t)t2 * L.W + w] & um & ~amb & ~A;
}

struct TwoEval {
    bool swap, dir, ok;
    int c1, c2, t1, t2;   // post-swap clade node ids / table positions
};

// set_synteny_two + apply_lgt_checks for one option (waafle_orgscorer.py:511-545, 678-744).
__device__ __noinline__ void eval_two(const Level &L, const DevTax &tax, const DevParams &P, int ta, int tb,
                                      TwoEval &ev) {
    const u64 *mamb = L.mk[P.amb_sel], *msis = L.mk[P.sis_sel];
    const bool unk = L.cl_id[ta] == tax.unknown || L.cl_id[tb] == tax.unknown;
    bool swap = false;
#pragma unroll 1
    for (int w = 0; w < L.W; ++w) {   // "^[^A]*B": first clear letter is B -> swap
        u64 A, B, amb;
        letters(L, mamb, unk, ta, tb, w, A, B, amb);
        u64 ab = A | B;
        if (ab) {
            u64 low = ab & (~ab + 1);
            swap = (B & low) != 0;
            break;
        }
    }
    ev.swap = swap;
    ev.t1 = swap ? tb : ta;
    ev.t2 = swap ? ta : tb;
    ev.c1 = L.cl_id[ev.t1];
    ev.c2 = L.cl_id[ev.t2];
    // one pass over the loci: lengths, counts, "^A+B+A+$" on the non-ignored letters
    long long total_len = 0, amb_len = 0;
    int nA = 0, nB = 0, state = 0;
#pragma unroll 1
    for (int w = 0; w < L.W; ++w) {
        u64 A, B, amb;
        letters(L, mamb, unk, ta, tb, w, A, B, amb);
        if (swap) { u64 t = A; A = B; B = t; }
        nA += __popcll(A);
        nB += __popcll(B);
        u64 bits = L.um[w];
        while (bits) {
            int b = __ffsll((long long)bits) - 1;
            bits &= bits - 1;
            u64 m = 1ull << b;
            int len = L.l_len[w * 64 + b];
            if (A & m) {
                total_len += len;
                state = (state == 0 || state == 1) ? 1 : (state == 2 || state == 3) ? 3 : -1;
            } else if (B & m) {
                total_len += len;
                state = (state == 1 || state == 2) ? 2 : -1;
            } else {
                if (amb & m) { total_len += len; amb_len += len; }
                state = -1;
            }
        }
    }
    ev.dir = state == 3;
    bool ok = true;
    if (total_len > 0 && (double)amb_len / (double)total_len > P.p.ambiguous_fraction) ok = false;
    if (P.p.clade_genes >= 0 && min(nA, nB) < P.p.clade_genes) ok = false;
    if (P.p.clade_leaves >= 0) {
        int lc = ev.dir ? tax.leaf_count[ev.c2] : min(tax.leaf_count[ev.c1], tax.leaf_count[ev.c2]);
        if (lc < P.p.clade_leaves) ok = false;
    }
    if (P.p.sister_penalty != 0 && ok) {
        const int p1 = tax.parent[ev.c1], p2 = tax.parent[ev.c2];
#pragma unroll 1
        for (int t = 0; t < L.T && ok; ++t) {
            const int px = L.cl_par[t];
            const bool s1 = px == p1, s2 = (px == p2) && !ev.dir;
            if (!s1 && !s2) continue;
            if (t == ev.t1 || t == ev.t2) continue;
            for (int w = 0; w < L.W; ++w) {
                u64 A, B, amb;
                letters(L, mamb, unk, ta, tb, w, A, B, amb);
                if (swap) { u64 tt = A; A = B; B = tt; }
                u64 ms = msis[(size_t)t * L.W + w];
                // a B locus is penalised by clade1's sisters, an A locus by clade2's
                if ((s1 && (ms & B)) || (s2 && (ms & A))) { ok = false; break; }
            }
        }
    }
    ev.ok = ok;
}

__device__ __noinline__ bool pair_pass(const Level &L, int t1, int t2) {
    bool pass = true;   // crit >= k2  <=>  every non-ignored locus has s1 >= k2 or s2 >= k2
#pragma unroll 1
    for (int w = 0; w < L.W; ++w)
        pass &= ((L.mk[1][(size_t)t1 * L.W + w] | L.mk[1][(size_t)t2 * L.W + w]) & L.um[w]) == L.um[w];
    return pass;
}

__device__ __noinline__ void pair_decode(long long p, int n, int &i, int &j) {
    // pairs enumerated i-major: (0,1),(0,2),...,(0,n-1),(1,2),...; offset(i) = i*(2n-i-1)/2
    double nn = 2.0 * n - 1.0;
    long long ii = (long long)floor((nn - sqrt(nn * nn - 8.0 * (double)p)) * 0.5);
    if (ii < 0) ii = 0;
    if (ii > n - 2) ii = n - 2;
    while (ii > 0 && ii * (2LL * n - ii - 1) / 2 > p) --ii;
    while ((ii + 1) * (2LL * n - ii - 2) / 2 <= p) ++ii;
    i = (int)ii;
    j = (int)(p - ii * (2LL * n - ii - 1) / 2) + i + 1;
}

// hit x locus test after the scov filter: strand / calc_overlap >= --min-overlap
// (waafle_orgscorer.py:365-367, utils.py:487-500)
__device__ __noinline__ bool hit_matches(const DevParams &P, int hmin, int hmax, signed char hs, int lmin, int llen,
                                         signed char ls) {
    if (P.p.stranded && hs != ls) return false;
    int lmax = lmin + llen - 1;
    double ov = 0.0;   // utils.py:492-499
    if (!(lmin > hmax || hmin > lmax))
        ov = (double)(min(hmax, lmax) - max(hmin, lmin) + 1) / (double)min(hmax - hmin + 1, llen);
    return ov >= P.p.min_overlap;
}

// site slice [s1, e1) a matched hit raises on a locus of length llen: the python slice [h1 : h2+1] of score_hit
// (waafle_orgscorer.py:376-382), including the wrap of a negative stop; e1 == s1 for an empty slice
__device__ __forceinline__ void hit_slice(int hmin, int hmax, int lmin, int llen, int &s1, int &e1) {
    s1 = max(0, hmin - lmin);
    e1 = min(llen - 1, hmax - lmin) + 1;
    if (e1 < 0) e1 = max(0, e1 + llen);
    s1 = min(s1, llen);
    if (e1 < s1) e1 = s1;
}


}  // namespace
}  // namespace wfl
