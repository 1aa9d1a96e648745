// The EXACT orgscorer path as a pipeline of small kernels, one warp per contig in every kernel.  It reproduces
// numpy's pairwise summation bit for bit; it scores the contigs the fused fast-path kernel (wfl_fast.cu) hands
// back (guard band tripped, or too large for its shared-memory slice) and everything under WFL_K2=exact.
//
//   wfl_pipe_prepare : K1 match + record emission, K3 annotations, base order, distinct-clade table
//                      (the only kernel that streams the hit SoA from HBM)
//   wfl_pipe_regroup : K5 regroup (stable multisplit by clade rank, group table)
//   wfl_pipe_k2hist / k2scan / k2scatter / k2 : K2 envelope integrals (gene score per (clade, locus) group) over
//                      the sub-batch's group list, counting-sorted so that a warp's lanes share a leaf plan
//   wfl_pipe_masks   : K4 weak loci, clade rows + gene bitmasks
//   wfl_pipe_one     : K6 one-clade search + meld; unresolved contigs go to the two-clade list
//   wfl_pipe_two     : K7/K8 two-clade search, meld, LGT filters; undecided contigs go to the lift list
//   wfl_pipe_lift    : K9 stop-or-lift (K5 lift of the clade table; next level's list)
//
// regroup/K2/masks/one/two/lift are launched once per taxonomy level over device-side work lists (no host sync in
// the level loop; an empty list makes the launch a no-op).  Between kernels a contig's state lives
// in a global workspace pool (regions A: loci, B: records + clade table, C: per-level arrays), carved
// by the same deterministic bump arena in every kernel.  Why small kernels: as one kernel this code is bound
// by instruction fetch (profiles/r1_final_score_kernel_ncu.txt); here every kernel's hot code fits the SM
// instruction cache and all warps of an SM run the same phase.
#include "wfl_warp_common.cuh"

namespace wfl {

namespace {

// per-phase cycle counters (wfl_stats.phase_cycles): compiled in only with -DWFL_PROFILE
#ifdef WFL_PROFILE
#define PH_BEGIN const long long t_start = clock64()
#define PH_END(i) do { if (lane == 0) atomicAdd(&a.ctr->phase_cycles[i], (unsigned long long)(clock64() - t_start)); } while (0)
#else
#define PH_BEGIN do { } while (0)
#define PH_END(i) do { } while (0)
#endif

#ifndef WFL_PIPE_CPSM
#define WFL_PIPE_CPSM 32   // resident single-warp CTAs per SM the pipeline kernels are compiled for
#endif
// The small kernels (regroup, masks, one-clade, lift) wait on dependent workspace loads; they can be compiled
// with several independent warps per CTA to pass the 32-CTAs-per-SM limit (more warps, fewer registers each).
#ifndef WFL_LAT_WPC
#define WFL_LAT_WPC 1      // warps per CTA of the latency-bound kernels
#endif
#ifndef WFL_LAT_CPSM
#define WFL_LAT_CPSM 32    // their resident CTAs per SM
#endif

// Linear bump arena over one workspace region: region sizes are exact (loci_bytes / record_bytes) or
// bounds (level_bytes), so carving is a pointer increment plus one capacity compare.
struct LinArena {
    char *base;
    size_t cap, used;
    bool ok;
    template <class T>
    __device__ __forceinline__ T *get(size_t n) {
        T *p = reinterpret_cast<T *>(base + used);
        used += (n * sizeof(T) + 15) & ~size_t(15);
        ok = ok && used <= cap;
        return p;
    }
};

#define DECL_LOCI                                                                                   \
    int *l_lo = arA.get<int>(Graw), *l_len = arA.get<int>(Graw), *l_raw = arA.get<int>(Graw);       \
    int *l_base = arA.get<int>(Graw + 2);                                                           \
    const u16 **l_plan = arA.get<const u16 *>(Graw + 1);                                            \
    int *l_nleaf = arA.get<int>(Graw + 1);                                                          \
    signed char *l_str = arA.get<signed char>(Graw);                                                \
    u32 *l_k8 = arA.get<u32>(Graw + 1);

#define DECL_RECORDS                                                                                \
    u16 *plan_fb = ar.get<u16>(np_tot);                                                             \
    double *r_v = ar.get<double>(M);                                                                \
    int *r_a = ar.get<int>(M), *r_b = ar.get<int>(M), *r_t = ar.get<int>(M), *r_loc = ar.get<int>(M), \
        *r_hit = S > 0 ? ar.get<int>(M) : nullptr;                                                  \
    int *base_ord = ar.get<int>(M);                                                                 \
    double *maxv = ar.get<double>(G);                                                               \
    u64 *maxb = ar.get<u64>(G);                                                                     \
    u8 *ign = ar.get<u8>(G + 1);                                                                    \
    u64 *um = ar.get<u64>(W);                                                                       \
    u64 *annb = S > 0 ? ar.get<u64>((size_t)G * S) : nullptr;                                       \
    int *annw = S > 0 ? ar.get<int>((size_t)G * S) : nullptr;                                       \
    int *cl_id = ar.get<int>(M + 2);                                                                \
    int *ord = ar.get<int>(M);                                                                      \
    int *map_t = ar.get<int>(M + 2);                                                                \
    u8 *fo = ar.get<u8>(M + 2);

#define DECL_CUR                                                                                    \
    int *cur = al.get<int>(T + 2);                                                                  \
    int *s_a = al.get<int>(M), *s_b = al.get<int>(M);                                               \
    double *s_v = al.get<double>(M);

#define DECL_GROUPS                                                                                 \
    double *g_score = al.get<double>(Ngrp);                                                         \
    int *g_rs = al.get<int>(Ngrp + 1), *g_re = al.get<int>(Ngrp + 1), *g_loc = al.get<int>(Ngrp),   \
        *g_t = al.get<int>(Ngrp), *gs = al.get<int>(ng + 1), *g_perm = al.get<int>(Ngrp),           \
        *gcur = al.get<int>(2 * G + 2);

#define DECL_CLADES                                                                                 \
    int *cl_go = al.get<int>(T + 1), *cand = al.get<int>(T);                                        \
    double *cl_rank = al.get<double>(T), *cl_crit = al.get<double>(T);                              \
    u8 *cl_opt = al.get<u8>(T), *memA = al.get<u8>(T), *memB = al.get<u8>(T);                       \
    u64 *mk0 = al.get<u64>((size_t)T * W), *mk1 = al.get<u64>((size_t)T * W),                       \
        *mk2 = al.get<u64>((size_t)T * W);                                                          \
    u64 *bestm = al.get<u64>(3 * (size_t)W);                                                        \
    int *cl_par = al.get<int>(T);                                                                   \
    Level *Lp = al.get<Level>(1);

__device__ __forceinline__ size_t al16(size_t b) { return (b + 15) & ~size_t(15); }

// exact size of region A (the DECL_LOCI arrays)
__device__ __forceinline__ size_t loci_bytes(int Graw) {
    return 3 * al16(4 * (size_t)Graw) + al16(4 * ((size_t)Graw + 2)) + al16(8 * ((size_t)Graw + 1)) +
           2 * al16(4 * ((size_t)Graw + 1)) + al16((size_t)Graw);
}
// region B: DECL_RECORDS exactly, plus the temporary hash table of the clade-table build
__device__ __forceinline__ size_t record_bytes(int M, int G, int W, int S, int np_tot, int nwords, size_t *persist) {
    size_t m = (size_t)M, g = (size_t)G;
    size_t p = al16(2 * (size_t)np_tot) + al16(8 * m) + 4 * al16(4 * m) + (S > 0 ? al16(4 * m) : 0) + al16(4 * m) +
               2 * al16(8 * g) + al16(g + 1) + al16(8 * (size_t)W) +
               (S > 0 ? al16(8 * g * S) + al16(4 * g * S) : 0) + al16(4 * (m + 2)) + al16(4 * m) + al16(4 * (m + 2)) +
               al16(m + 2);
    *persist = p;
    size_t cap = 64;
    while (cap < 2 * (m + 1)) cap <<= 1;
    size_t hash_tmp = 2 * al16(4 * cap) + al16(4 * (m + 1)) + 64;
    size_t bitmap_tmp = nwords <= BITMAP_MAX_WORDS ? 2 * al16(4 * ((size_t)nwords + 1)) + 64 : 0;
    return p + (nwords <= BITMAP_MAX_WORDS ? bitmap_tmp : hash_tmp);
}
// region C: bound on the per-level arrays once the number of distinct clades T is known
__device__ __forceinline__ size_t level_bytes(int T, int M, int G, int W, int nwords) {
    size_t t = (size_t)T, ngb = (size_t)min((long long)M, (long long)T * G) + (size_t)G + 1;
    return al16(4 * (t + 2)) + 16 * (size_t)M + 48 + 40 * ngb + al16(4 * (2 * (size_t)G + 2)) + 160 + 27 * t + 24 * (size_t)W * t + 24 * (size_t)W +
           256 + sizeof(Level) + al16(4 * (t + 1)) + 4 * t + 16 * 25 + 6144 +
           (((size_t)nwords <= (size_t)BITMAP_MAX_WORDS) ? 8 * (size_t)nwords + 96 : 0);
}

struct ContigOut {
    int call, dir, c1, c2, lca, b1, b2, na, nb, status, lifts;
    long long mem;
    double crit, rank;
};

__device__ __noinline__ void write_result(const PipeArgs &a, long long c, const ContigOut &r) {
    if (r.status == 1) {
        atomicAdd(&a.ctr->n_overflow, 1ull);
    }
    if (r.status == 2) atomicAdd(&a.ctr->n_runaway, 1ull);
    if (r.status == 3) atomicAdd(&a.ctr->n_badinput, 1ull);
    a.o.call[c] = (uint8_t)r.call;
    a.o.direction[c] = (uint8_t)r.dir;
    a.o.lifts[c] = r.lifts;
    a.o.clade1[c] = r.c1;
    a.o.clade2[c] = r.c2;
    a.o.lca[c] = r.lca;
    a.o.best1[c] = r.b1;
    a.o.best2[c] = r.b2;
    a.o.crit[c] = r.crit;
    a.o.rank[c] = r.rank;
    a.o.n_mem_a[c] = r.na;
    a.o.n_mem_b[c] = r.nb;
    a.o.mem_pos[c] = r.mem;
    a.o.status[c] = (uint8_t)r.status;
}

#define RESULT_LOCALS                                                                               \
    int r_call = WFL_CALL_UNCLASSIFIED, r_dir = 0, r_c1 = -1, r_c2 = -1, r_lca = -1, r_b1 = -1, r_b2 = -1, \
        r_na = 0, r_nb = 0, r_status = 0;                                                           \
    long long r_mem = 0;                                                                            \
    double r_crit = 0.0, r_rank = 0.0;                                                              \
    (void)r_status;

#define EMIT_RESULT(status_)                                                                        \
    do {                                                                                            \
        if (lane == 0) {                                                                            \
            ContigOut ro{r_call, r_dir, r_c1, r_c2, r_lca, r_b1, r_b2, r_na, r_nb, (status_), lifts, r_mem, r_crit, \
                         r_rank};                                                                   \
            write_result(a, c, ro);                                                                 \
            a.ctg[c].state = PIPE_DONE;                                                             \
        }                                                                                           \
    } while (0)

// fetch the next work item of a launch (lane 0 pops, the warp follows)
__device__ __forceinline__ long long pop_work(unsigned long long *wq, const int *list, const int *count, int lane) {
    long long c = -1;
    if (lane == 0) {
        unsigned long long w = atomicAdd(wq, 1ull);
        if ((long long)w < (long long)*count) c = list[w];
    }
    return __shfl_sync(FULL, c, 0);
}

// rebuild the arenas of a contig from its saved context (regions A+B persistent, B-leftover+C per level)
#define OPEN_CONTIG                                                                                 \
    const PipeCtg cx = a.ctg[c];                                                                    \
    const long long h0 = a.b.hit_off[c], l0 = a.b.locus_off[c];                                     \
    const int H = (int)(a.b.hit_off[c + 1] - h0), Graw = (int)(a.b.locus_off[c + 1] - l0);          \
    (void)H; (void)h0;                                                                              \
    const int G = cx.G, W = cx.W, M = cx.M, np_tot = cx.np_tot, iter = cx.iter;                     \
    int T = cx.T, lifts = cx.lifts;                                                                 \
    LinArena arA{a.pool + cx.offA, (size_t)cx.capA, 0, true};                                       \
    LinArena ar{a.pool + cx.offB, (size_t)cx.capB, 0, true};                                        \
    DECL_LOCI                                                                                       \
    DECL_RECORDS                                                                                    \
    LinArena al{a.pool + cx.offC, (size_t)cx.capC, 0, true};                                        \
    (void)l_lo; (void)l_base; (void)l_plan; (void)l_nleaf; (void)l_str; (void)l_k8; (void)plan_fb;  \
    (void)r_a; (void)r_b; (void)r_hit; (void)base_ord; (void)maxv; (void)annb; (void)annw; (void)map_t; (void)fo; \
    (void)r_v; (void)ord; (void)maxb; (void)iter;

}  // namespace

// ---------------------------------------------------------------------------------------------
// kernel 1: prepare
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32, WFL_PIPE_CPSM) wfl_pipe_prepare(const PipeArgs a) {
    const int lane = threadIdx.x;
    const DevParams &P = a.P;
    const DevTax &tax = a.t;
    const int S = P.p.n_systems;
    const bool spike = P.p.weak_loci == 2;
#pragma unroll 1
    for (;;) {
        long long c = -1;
        if (lane == 0) {
            unsigned long long w = atomicAdd(a.wq, 1ull);
            c = (long long)w < a.n_work ? (a.work_list ? (long long)a.work_list[w] : a.work_base + (long long)w) : -1;
        }
        c = __shfl_sync(FULL, c, 0);
        if (c < 0) break;
        PH_BEGIN;
        const long long h0 = a.b.hit_off[c], l0 = a.b.locus_off[c];
        const int H = (int)(a.b.hit_off[c + 1] - h0), Graw = (int)(a.b.locus_off[c + 1] - l0);
        RESULT_LOCALS
        bool bad_input = false, overflow = false;
        // region A
        const size_t capA = loci_bytes(Graw);
        unsigned long long offA = 0;
        if (lane == 0) offA = atomicAdd(a.pool_used, (unsigned long long)((capA + 255) & ~size_t(255)));
        offA = __shfl_sync(FULL, offA, 0);
        const bool fitsA = offA + capA <= a.pool_cap;
        LinArena arA{a.pool + (fitsA ? offA : 0), fitsA ? capA : 0, 0, true};
        LinArena ar{a.pool, 0, 0, true};
        DECL_LOCI
        if (!fitsA) arA.ok = false;
        overflow = !arA.ok;
        int G = 0;
#pragma unroll 1
        for (int base = 0; base < Graw && !overflow; base += 32) {
            int j = base + lane, flag = 0, lo = 0, len = 0;
            if (j < Graw) {
                int s = a.b.locus_start[l0 + j], e = a.b.locus_end[l0 + j];
                lo = min(s, e);
                len = max(s, e) - lo + 1;
                flag = (double)len >= P.p.min_gene_length;
                a.o.locus_flags[l0 + j] = flag ? WFL_LOCUS_RETAINED : 0;
                a.o.synteny[l0 + j] = 0;
#pragma unroll 1
                for (int s2 = 0; s2 < S; ++s2) a.o.ann_winner[(l0 + j) * S + s2] = -1;
            }
            u32 m = __ballot_sync(FULL, flag);
            if (flag) {
                int pos = G + __popc(m & lt_mask());
                l_lo[pos] = lo;
                l_len[pos] = len;
                l_raw[pos] = j;
                l_str[pos] = a.b.locus_strand[l0 + j];
            }
            G += __popc(m);
        }
        __syncwarp();
        __syncwarp();
        const int W = (G + 63) >> 6;
        int lifts = H > 0 ? P.p.jump_taxonomy : 0;
        int M = 0, np_tot = 0, T = 0;
        bool active = false;
        if (!overflow && H > 0 && G > 0) {
            // ---- leaf plans: host-built table for lengths <= plan_nmax, in-kernel build beyond -------
#pragma unroll 1
            for (int i = lane; i <= G + 1; i += 32) l_base[i] = 0;
            np_tot = 0;
#pragma unroll 1
            for (int base = 0; base < G; base += 32) {
                int i = base + lane, np = (i < G && l_len[i] > a.plan_nmax) ? plan_cap(l_len[i]) : 0, tot;
                int ex = warp_excl_scan(np, tot);
                if (i < G) l_nleaf[i] = np_tot + ex;
                np_tot += tot;
            }
            __syncwarp();
            // ---- K1 pass 1: matches per locus (ballot counts) --------------------------------------
            const bool all_match = P.p.min_overlap <= 0.0;   // disjoint pairs "overlap" 0 >= min_overlap
#pragma unroll 1
            for (int base = 0; base < H; base += 32) {
                int h = base + lane;
                bool hok = false;
                int hmin = 0, hmax = 0;
                signed char hs = 0;
                if (h < H) {
                    hok = hit_scov_ok(a.b, h0 + h, P.p.min_scov);   // waafle_orgscorer.py:362
                    int q1, q2;
                    hit_span(a.b, h0 + h, q1, q2);
                    hmin = min(q1, q2);
                    hmax = max(q1, q2);
                    hs = hit_strand_of(a.b, h0 + h);
                }
                if (!__any_sync(FULL, hok)) continue;
#pragma unroll 1
                for (int i = 0; i < G; ++i) {
                    const int lmin = l_lo[i], llen = l_len[i];
                    bool cand = hok && (all_match || !(lmin > hmax || hmin > lmin + llen - 1));
                    if (!__any_sync(FULL, cand)) continue;
                    u32 m = __ballot_sync(FULL, cand && hit_matches(P, hmin, hmax, hs, lmin, llen, l_str[i]));
                    if (lane == 0 && m) l_base[i + 1] += __popc(m);
                }
            }
            __syncwarp();
            M = 0;
#pragma unroll 1
            for (int base = 0; base < G; base += 32) {   // exclusive scan -> record base of each locus
                int i = base + lane, cnt = i < G ? l_base[i + 1] : 0, tot;
                int ex = warp_excl_scan(cnt, tot);
                __syncwarp();
                if (i < G) l_base[i + 1] = M + ex;   // cursor of locus i lives in l_base[i+1] during the fill
                M += tot;
            }
            __syncwarp();
            // region B
            size_t persist = 0;
            const size_t capB = record_bytes(M, G, W, S, np_tot, (tax.n_nodes + 31) >> 5, &persist);
            unsigned long long offB = 0;
            if (lane == 0) offB = atomicAdd(a.pool_used, (unsigned long long)((capB + 255) & ~size_t(255)));
            offB = __shfl_sync(FULL, offB, 0);
            if (offB + capB <= a.pool_cap) {
                ar.base = a.pool + offB;
                ar.cap = capB;
            } else {
                ar.ok = false;
            }
            DECL_RECORDS
            overflow = !ar.ok;
            if (!overflow) {
#pragma unroll 1
                for (int i = lane; i < G; i += 32) {
                    const int len = l_len[i];
                    if (len <= a.plan_nmax) {
                        const PlanEntry pe = a.plan_index[len];
                        l_plan[i] = a.plan_data + pe.off;
                        l_nleaf[i] = (int)pe.nleaf;
                        l_k8[i] = pe.k8;
                    } else {
                        u16 *dst = plan_fb + l_nleaf[i];
                        l_plan[i] = dst;
                        l_nleaf[i] = build_plan(len, dst, reinterpret_cast<u8 *>(&l_k8[i]));
                    }
                }
#pragma unroll 1
                for (int i = lane; i < G * S; i += 32) { annb[i] = 0; annw[i] = -1; }
                __syncwarp();
                // ---- K1 pass 2: emit records (score_hit, waafle_orgscorer.py:371-382) -------------
#pragma unroll 1
                for (int base = 0; base < H; base += 32) {
                    int h = base + lane;
                    bool hok = false;
                    int hmin = 0, hmax = 0, cl = 0;
                    signed char hs = 0;
                    double sc = 0.0;
                    u32 sys = 0;
                    if (h < H) {
                        hok = hit_scov_ok(a.b, h0 + h, P.p.min_scov);
                        int q1, q2;
                        hit_span(a.b, h0 + h, q1, q2);
                        hmin = min(q1, q2);
                        hmax = max(q1, q2);
                        hs = hit_strand_of(a.b, h0 + h);
                    }
                    if (!__any_sync(FULL, hok)) continue;
                    if (hok) {
                        cl = hit_taxon_of(a.b, h0 + h);
                        if ((u32)cl >= (u32)tax.n_nodes) { cl = tax.root; bad_input = true; }
#pragma unroll 1
                        for (int j = 0; j < P.p.jump_taxonomy; ++j) cl = tax.parent[cl];
                        sc = a.b.hit_score[h0 + h];
                        if (S > 0) sys = hit_sysmask_of(a.b, h0 + h);
                    }
#pragma unroll 1
                    for (int i = 0; i < G; ++i) {
                        const int lmin = l_lo[i], len = l_len[i];
                        bool cand = hok && (all_match || !(lmin > hmax || hmin > lmin + len - 1));
                        if (!__any_sync(FULL, cand)) continue;
                        bool mt = cand && hit_matches(P, hmin, hmax, hs, lmin, len, l_str[i]);
                        u32 m = __ballot_sync(FULL, mt);
                        if (!m) continue;
                        int cur = l_base[i + 1];
                        if (mt) {
                            int slot = cur + __popc(m & lt_mask());
                            int s1, e1;
                            hit_slice(hmin, hmax, lmin, len, s1, e1);
                            r_v[slot] = sc;
                            r_a[slot] = s1;
                            r_b[slot] = e1;
                            r_t[slot] = cl;
                            r_loc[slot] = i;
                            if (S > 0) {
                                r_hit[slot] = h;
                                // K3 phase 1: max annotated score per (locus, system)
                                u32 ms = sys;
                                if (ms && sc >= P.ann_thr) {
                                    u64 sb = dbits(sc);
                                    while (ms) {
                                        int s2 = __ffs(ms) - 1;
                                        ms &= ms - 1;
                                        atomicMax(&annb[(size_t)i * S + s2], sb);
                                    }
                                }
                            }
                        }
                        __syncwarp();
                        if (lane == 0) l_base[i + 1] = cur + __popc(m);
                        __syncwarp();
                    }
                }
                __syncwarp();
                // after the fill, l_base[i+1] == end of locus i == start of locus i+1; l_base[0] == 0
                if (S > 0) {
                    // K3 phase 2: the LAST hit (file order) attaining the max wins (:389, '>=')
#pragma unroll 1
                    for (int r = lane; r < M; r += 32) {
                        u32 ms = hit_sysmask_of(a.b, h0 + r_hit[r]);
                        double sc = r_v[r];
                        if (ms && sc >= P.ann_thr) {
                            u64 sb = dbits(sc);
                            while (ms) {
                                int s2 = __ffs(ms) - 1;
                                ms &= ms - 1;
                                if (annb[(size_t)r_loc[r] * S + s2] == sb)
                                    atomicMax(&annw[(size_t)r_loc[r] * S + s2], r_hit[r]);
                            }
                        }
                    }
                    __syncwarp();
#pragma unroll 1
                    for (int i = lane; i < G * S; i += 32) {
                        int w = annw[i];
                        a.o.ann_winner[(l0 + l_raw[i / S]) * S + (i % S)] = w >= 0 ? (int)(h0 + w) : -1;
                    }
                }
                {
                    // ---- level-invariant base order (built once):
                    // inside each locus, records by descending score
                    // (rank by counting; ties keep emission order).  Every later regrouping is a STABLE
                    // split of this sequence, so each (clade, locus) group arrives score-descending and
                    // the envelope scan can stop at the first record covering a site.
#pragma unroll 1
                    for (int r = lane; r < M; r += 32) {
                        const int loc = r_loc[r], s0 = l_base[loc], s1 = l_base[loc + 1];
                        const double v = r_v[r];
                        int rk = 0;
#pragma unroll 4
                        for (int q = s0; q < s1; ++q) {
                            double vq = r_v[q];
                            rk += (vq > v) || (vq == v && q < r);
                        }
                        base_ord[s0 + rk] = r;
                    }
                    __syncwarp();
                }
                const int nwords = (tax.n_nodes + 31) >> 5;
                if (nwords <= BITMAP_MAX_WORDS) {
                    // small taxonomies: presence bitmap over the node indices; the rank of a clade among the
                    // contig's clades is a prefix popcount (ascending node index == ascending name)
                    u32 *bm = ar.get<u32>(nwords);
                    int *bpre = ar.get<int>(nwords + 1);
                    if (!ar.ok) overflow = true;
                    if (!overflow) {
#pragma unroll 1
                        for (int w = lane; w < nwords; w += 32) bm[w] = 0;
                        __syncwarp();
#pragma unroll 1
                        for (int r = lane; r < M + (spike ? 1 : 0); r += 32) {
                            const int key = r < M ? r_t[r] : tax.unknown;
                            atomicOr(&bm[key >> 5], 1u << (key & 31));
                        }
                        __syncwarp();
#pragma unroll 1
                        for (int base = 0; base < nwords; base += 32) {
                            const int w = base + lane;
                            const u32 bits = w < nwords ? bm[w] : 0u;
                            int tot, ex = warp_excl_scan(__popc(bits), tot);
                            if (w < nwords) {
                                int pos = T + ex;
                                bpre[w] = pos;
                                u32 b = bits;
                                while (b) {
                                    cl_id[pos++] = (w << 5) + __ffs(b) - 1;
                                    b &= b - 1;
                                }
                            }
                            T += tot;
                        }
                        __syncwarp();
#pragma unroll 1
                        for (int r = lane; r < M; r += 32) {
                            const int key = r_t[r];
                            r_t[r] = bpre[key >> 5] + __popc(bm[key >> 5] & ((1u << (key & 31)) - 1u));
                        }
                        __syncwarp();
                    }
                } else {
                    int cap = 64;
                    while (cap < 2 * (M + 1)) cap <<= 1;
                    int *hk = ar.get<int>(cap), *hv = ar.get<int>(cap);
                    int *dl = ar.get<int>(M + 1);
                    if (!ar.ok) overflow = true;
                    if (!overflow) {
#pragma unroll 1
                        for (int i = lane; i < cap; i += 32) hk[i] = -1;
                        __syncwarp();
#pragma unroll 1
                        for (int r = lane; r < M + (spike ? 1 : 0); r += 32) {
                            int key = r < M ? r_t[r] : tax.unknown;
                            u32 slot = ((u32)key * 2654435761u) & (cap - 1);
#pragma unroll 1
                            for (;;) {
                                int old = atomicCAS(&hk[slot], -1, key);
                                if (old == -1 || old == key) break;
                                slot = (slot + 1) & (cap - 1);
                            }
                            if (r < M) r_t[r] = (int)slot;
                        }
                        __syncwarp();
#pragma unroll 1
                        for (int base = 0; base < cap; base += 32) {   // compact the distinct keys
                            int i = base + lane;
                            bool f = hk[i] >= 0;
                            u32 m = __ballot_sync(FULL, f);
                            if (f) dl[T + __popc(m & lt_mask())] = i;
                            T += __popc(m);
                        }
                        __syncwarp();
#pragma unroll 1
                        for (int j = lane; j < T; j += 32) map_t[j] = hk[dl[j]];   // compact key list
                        __syncwarp();
#pragma unroll 1
                        for (int j = lane; j < T; j += 32) {   // rank = #distinct keys below
                            int key = map_t[j], rk = 0;
#pragma unroll 4
                            for (int q = 0; q < T; ++q) rk += map_t[q] < key;
                            hv[dl[j]] = rk;
                            cl_id[rk] = key;
                        }
                        __syncwarp();
#pragma unroll 1
                        for (int r = lane; r < M; r += 32) r_t[r] = hv[r_t[r]];
                        __syncwarp();
                    }
                }
            }
            const bool bad = __any_sync(FULL, bad_input);
            if (!overflow && !bad) {
                // region C: per-level arrays, sized now that T is known
                const size_t capC = level_bytes(T, M, G, W, (tax.n_nodes + 31) >> 5);
                unsigned long long offC = 0;
                if (lane == 0) offC = atomicAdd(a.pool_used, (unsigned long long)((capC + 255) & ~size_t(255)));
                offC = __shfl_sync(FULL, offC, 0);
                if (offC + capC > a.pool_cap) {
                    overflow = true;
                } else if (lane == 0) {
                    PipeCtg cx;
                    cx.offA = offA; cx.offB = offB; cx.offC = offC;
                    cx.capA = (unsigned)capA; cx.capB = (unsigned)capB; cx.capC = (unsigned)capC;
                    cx.G = G; cx.W = W; cx.M = M; cx.T = T; cx.np_tot = np_tot; cx.lifts = lifts; cx.iter = 0;
                    cx.Ngrp = cx.ng = cx.nlt = cx.nu = cx.nun = cx.hasroot = 0; cx.t_unk = -1;
                    cx.state = PIPE_ACTIVE;
                    a.ctg[c] = cx;
                    int slot = atomicAdd(a.cnt_act, 1);
                    a.list_act[slot] = (int)c;
                    atomicAdd(&a.ctr->matched_pairs, (unsigned long long)M);
                }
                active = !overflow;
            }
        }
        if (__any_sync(FULL, bad_input)) { overflow = false; r_status = 3; }
        if (!active) {
            if (overflow) r_status = 1;
            EMIT_RESULT(r_status);
        }
        PH_END(0);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 2a: regroup (K5) -- records in (clade, locus) group order, group table
// ---------------------------------------------------------------------------------------------
// The scoring step is cut in three kernels (regroup | K2 | masks) for the same reason the pipeline
// exists: as one kernel it ran with an SM instruction-cache hit rate of 87 % and the GPC instruction
// cache at 92 % of its request throughput (profiles/r1_final2_pipeline_kernels_ncu.txt).
__global__ void __launch_bounds__(32 * WFL_LAT_WPC, WFL_LAT_CPSM) wfl_pipe_regroup(const PipeArgs a) {
    const int lane = threadIdx.x & 31;
    const DevParams &P = a.P;
    const DevTax &tax = a.t;
    const int S = P.p.n_systems;
    const bool spike = P.p.weak_loci == 2;
#pragma unroll 1
    for (;;) {
        const long long c = pop_work(a.wq, a.list_act, a.cnt_act, lane);
        if (c < 0) break;
        PH_BEGIN;
        OPEN_CONTIG
        RESULT_LOCALS
        bool overflow = false;
        int Ngrp = 0, ng = 0, nlt = 0, nu = 0, t_unk = -1;
        long long n_groups = 0;
#pragma unroll 1
        for (int once = 0; once < 1; ++once) {
            // ---- regroup: stable multisplit of the locus-major records by clade rank ------
            DECL_CUR
            if (!al.ok) { overflow = true; break; }
            warp_multisplit(M, T, r_t, base_ord, cur, ord);
            __syncwarp();
            // slices and scores copied into group order: the envelope scans read them contiguously
#pragma unroll 1
            for (int r = lane; r < M; r += 32) {
                const int i = ord[r];
                s_a[r] = r_a[i];
                s_b[r] = r_b[i];
                s_v[r] = r_v[i];
            }
            // groups = maximal runs of equal (clade rank, locus) in ord
            t_unk = -1;
            if (spike) {
                int lo = 0, hi = T;   // cl_id ascending: binary search for Unknown
                while (lo < hi) {
                    int mid = (lo + hi) >> 1;
                    if (cl_id[mid] < tax.unknown) lo = mid + 1; else hi = mid;
                }
                t_unk = lo;   // present by construction (inserted before ranking / kept by lifts)
            }
            ng = 0; nlt = 0; nu = 0;
#pragma unroll 1
            for (int base = 0; base < M; base += 32) {
                int r = base + lane;
                bool f = false;
                int t = 0;
                if (r < M) {
                    int i = ord[r];
                    t = r_t[i];
                    f = r == 0 || t != r_t[ord[r - 1]] || r_loc[i] != r_loc[ord[r - 1]];
                }
                ng += __popc(__ballot_sync(FULL, f));
                if (spike) {
                    nlt += __popc(__ballot_sync(FULL, f && t < t_unk));
                    nu += __popc(__ballot_sync(FULL, f && t == t_unk));
                }
            }
            Ngrp = spike ? ng - nu + G : ng;
            n_groups += Ngrp;
            DECL_GROUPS
            if (!al.ok) { overflow = true; break; }
            int gbase = 0;
#pragma unroll 1
            for (int base = 0; base < M; base += 32) {
                int r = base + lane;
                bool f = false;
                int t = 0, loc = 0;
                if (r < M) {
                    int i = ord[r];
                    t = r_t[i];
                    loc = r_loc[i];
                    f = r == 0 || t != r_t[ord[r - 1]] || loc != r_loc[ord[r - 1]];
                }
                u32 m = __ballot_sync(FULL, f);
                if (f) {
                    int gid = gbase + __popc(m & lt_mask()), dst = gid;
                    if (spike) dst = t < t_unk ? gid : (t == t_unk ? -1 : gid - nu + G);
                    gs[gid] = r;
                    if (dst >= 0) {
                        g_rs[dst] = r;
                        g_re[dst] = gid;   // patched to the end position below
                        g_loc[dst] = loc;
                        g_t[dst] = t;
                    }
                }
                gbase += __popc(m);
            }
            if (lane == 0) gs[ng] = M;
            __syncwarp();
#pragma unroll 1
            for (int g = lane; g < Ngrp; g += 32)
                if (!(spike && g >= nlt && g < nlt + G)) g_re[g] = gs[g_re[g] + 1];
            if (spike)
                for (int i = lane; i < G; i += 32) {
                    g_rs[nlt + i] = -1;
                    g_loc[nlt + i] = i;
                    g_t[nlt + i] = t_unk;
                }
#pragma unroll 1
            for (int i = lane; i < G; i += 32) maxb[i] = dbits(0.0);
            __syncwarp();
            {
                // ---- K2 work items: one descriptor per group with records, appended to the sub-batch's list
                const int nreal = spike ? Ngrp - G : Ngrp;   // the G spiked Unknown rows carry no records
                // reserve nreal slots with ONE atomic add (a compare-and-swap loop on this counter serialises the
                // whole grid).  A contig that does not fit fills its in-range slots with null items, which the K2
                // kernel skips, and is replayed by the warp kernel.
                unsigned long long dbase = 0;
                if (lane == 0) dbase = atomicAdd(&a.k2_meta->count, (unsigned long long)nreal);
                dbase = __shfl_sync(FULL, dbase, 0);
                if (dbase + (unsigned long long)nreal > a.k2_cap) {
                    K2Desc d{};
                    unsigned int nfill = 0;
#pragma unroll 1
                    for (unsigned long long i = dbase + lane; i < a.k2_cap; i += 32) {
                        a.k2_desc[i] = d;
                        a.k2_keys[i] = 0u;
                        ++nfill;
                    }
                    (void)nfill;
                    overflow = true;
                    break;
                }
                int wbase = 0;
#pragma unroll 1
                for (int gb = 0; gb < Ngrp; gb += 32) {
                    const int g = gb + lane;
                    const bool f = g < Ngrp && g_rs[g] >= 0;
                    const u32 m = __ballot_sync(FULL, f);
                    if (f) {
                        const int loc = g_loc[g], rs = g_rs[g], re = g_re[g], nleaf = l_nleaf[loc];
                        const int kc = re - rs <= 1 ? 0 : (re - rs <= 3 ? 1 : (re - rs <= 8 ? 2 : 3));
                        const int key = (min(nleaf, 127) << 2) | kc;
                        K2Desc d;
                        d.sa = s_a; d.plan = l_plan[loc]; d.out = &g_score[g];
                        d.maxb = cl_id[g_t[g]] != tax.unknown ? &maxb[loc] : nullptr;
                        d.d_sb = (int)(s_b - s_a);
                        d.d_sv = (int)(reinterpret_cast<const char *>(s_v) - reinterpret_cast<const char *>(s_a));
                        d.rs = rs; d.re = re; d.n = l_len[loc]; d.nleaf = nleaf; d.k8 = l_k8[loc]; d.key = (unsigned)key;
                        if (kc == 0) {
                            // a single record travels inside the descriptor (73 % of the groups at cfg2): K2 then
                            // never touches the record arrays of a contig it knows nothing else about
                            d.sa = reinterpret_cast<const int *>((size_t)__double_as_longlong(s_v[rs]));
                            d.d_sb = s_a[rs];
                            d.d_sv = s_b[rs];
                        }
                        const unsigned long long slot = dbase + wbase + __popc(m & lt_mask());
                        a.k2_desc[slot] = d;
                        a.k2_keys[slot] = (unsigned)key;
                    }
                    wbase += __popc(m);
                }
            }
        }
        if (lane == 0) {
            atomicAdd(&a.ctr->groups, (unsigned long long)n_groups);
            atomicAdd(&a.ctr->levels, 1ull);
        }
        if (overflow) {
            EMIT_RESULT(1);
        } else if (lane == 0) {
            PipeCtg *cp = &a.ctg[c];
            cp->Ngrp = Ngrp; cp->ng = ng; cp->nlt = nlt; cp->nu = nu; cp->t_unk = t_unk;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// kernels 2b: K2 (envelope integral of every (clade, locus) group, numpy-pairwise-exact) over the sub-batch's GLOBAL group list.  Counting sort of the descriptors by
// (leaf count, record-count class), then lane per group: the lanes of a warp walk the same leaf plan
// whatever contig their group belongs to (per contig, lanes met different plans and a partly filled last
// round: 11 of 32 threads active per instruction).
// ---------------------------------------------------------------------------------------------
constexpr int K2_TILE = 4096;   // items per block pass of the counting sort (256 threads x 16)

// histogram of the sort keys: per-block counts in shared memory, one flush per block
__global__ void __launch_bounds__(256) wfl_pipe_k2hist(const PipeArgs a) {
    __shared__ unsigned int cnt[K2_KEYS];
    const unsigned long long n = a.k2_meta->count < a.k2_cap ? a.k2_meta->count : a.k2_cap;
    for (int k = threadIdx.x; k < K2_KEYS; k += 256) cnt[k] = 0;
    __syncthreads();
    for (unsigned long long i = (unsigned long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * 256)
        atomicAdd(&cnt[a.k2_keys[i] & (K2_KEYS - 1)], 1u);
    __syncthreads();
    for (int k = threadIdx.x; k < K2_KEYS; k += 256)
        if (cnt[k]) atomicAdd(&a.k2_meta->hist[k], cnt[k]);
}

__global__ void wfl_pipe_k2scan(const PipeArgs a) {
    __shared__ unsigned int part[K2_KEYS];
    const int t = threadIdx.x;   // K2_KEYS threads
    const unsigned int h = a.k2_meta->hist[t];
    part[t] = h;
    __syncthreads();
    for (int o = 1; o < K2_KEYS; o <<= 1) {
        unsigned int v = t >= o ? part[t - o] : 0u;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    a.k2_meta->cursor[t] = part[t] - h;
}

// scatter: a block ranks a tile of items per key in shared memory, reserves one range per key with a single
// global atomic, and writes the item indices to their sorted positions
__global__ void __launch_bounds__(256) wfl_pipe_k2scatter(const PipeArgs a) {
    __shared__ unsigned int cnt[K2_KEYS], base[K2_KEYS];
    const unsigned long long n = a.k2_meta->count < a.k2_cap ? a.k2_meta->count : a.k2_cap;
    for (unsigned long long t0 = (unsigned long long)blockIdx.x * K2_TILE; t0 < n; t0 += (unsigned long long)gridDim.x * K2_TILE) {
        for (int k = threadIdx.x; k < K2_KEYS; k += 256) cnt[k] = 0;
        __syncthreads();
        unsigned int key[K2_TILE / 256], rk[K2_TILE / 256];
#pragma unroll
        for (int q = 0; q < K2_TILE / 256; ++q) {
            const unsigned long long i = t0 + (unsigned long long)q * 256 + threadIdx.x;
            key[q] = i < n ? (a.k2_keys[i] & (K2_KEYS - 1)) : 0xffffffffu;
            rk[q] = i < n ? atomicAdd(&cnt[key[q]], 1u) : 0u;
        }
        __syncthreads();
        for (int k = threadIdx.x; k < K2_KEYS; k += 256)
            if (cnt[k]) base[k] = atomicAdd(&a.k2_meta->cursor[k], cnt[k]);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < K2_TILE / 256; ++q) {
            const unsigned long long i = t0 + (unsigned long long)q * 256 + threadIdx.x;
            if (i < n) a.k2_order[base[key[q]] + rk[q]] = (unsigned int)i;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(32, WFL_PIPE_CPSM) wfl_pipe_k2(const PipeArgs a) {
    const int lane = threadIdx.x;
    const unsigned long long n = a.k2_meta->count < a.k2_cap ? a.k2_meta->count : a.k2_cap;
#pragma unroll 1
    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&a.k2_meta->take, 32ull);
        base = __shfl_sync(FULL, base, 0);
        if (base >= n) break;
        PH_BEGIN;
        const unsigned long long i = base + lane;
        if (i < n) {
            const K2Desc d = a.k2_desc[a.k2_order[i]];
            if (d.out != nullptr) {
            double sc;
            if ((d.key & 3u) == 0u) {   // single record, inline: slice [d_sb, d_sv), score in the bits of `sa`
                int a1 = d.d_sb, b1 = d.d_sv;
                double v1 = __longlong_as_double((long long)(size_t)d.sa);
                sc = group_mean(&a1, &b1, &v1, 0, 1, d.n, true, d.k8, d.plan, d.nleaf);
            } else {
                sc = group_mean(d.sa, d.sa + d.d_sb,
                                reinterpret_cast<const double *>(reinterpret_cast<const char *>(d.sa) + d.d_sv),
                                d.rs, d.re, d.n, true, d.k8, d.plan, d.nleaf);
            }
            *d.out = sc;
            if (d.maxb != nullptr) atomicMax(d.maxb, dbits(sc));   // waafle_orgscorer.py:409-411
            }
        }
        PH_END(3);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 2c: weak loci (K4), clade rows and gene bitmasks
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * WFL_LAT_WPC, WFL_LAT_CPSM) wfl_pipe_masks(const PipeArgs a) {
    const int lane = threadIdx.x & 31;
    const DevParams &P = a.P;
    const DevTax &tax = a.t;
    const int S = P.p.n_systems;
    const bool spike = P.p.weak_loci == 2;
#pragma unroll 1
    for (;;) {
        const long long c = pop_work(a.wq, a.list_act, a.cnt_act, lane);
        if (c < 0) break;
        if (a.ctg[c].state != PIPE_ACTIVE) continue;
        PH_BEGIN;
        OPEN_CONTIG
        RESULT_LOCALS
        const int Ngrp = cx.Ngrp, ng = cx.ng, nlt = cx.nlt;
        DECL_CUR
        DECL_GROUPS
        (void)cur; (void)s_a; (void)s_b; (void)s_v; (void)g_rs; (void)g_re; (void)gs; (void)g_perm; (void)gcur;
        (void)r_t; (void)r_loc;
        bool overflow = false, cont_ok = false;
        int nun = 0, hasroot = 0;
#pragma unroll 1
        for (int once = 0; once < 1; ++once) {
            // ---- K4: weak loci (waafle_orgscorer.py:412-427) ---------------------------------
#pragma unroll 1
            for (int i = lane; i < G; i += 32) {
                double mx = dbits_inv(maxb[i]);
                maxv[i] = mx;
                ign[i] = (P.p.weak_loci == 0) ? !(mx >= P.min_thr) : 0;
                if (spike) g_score[nlt + i] = 1.0 - mx;
            }
            if (lane == 0) ign[G] = 0;   // sentinel for ScoreSrc
            __syncwarp();
            nun = 0;
#pragma unroll 1
            for (int w = lane; w < W; w += 32) {
                u64 m = 0;
#pragma unroll 1
                for (int b = 0; b < 64 && w * 64 + b < G; ++b)
                    if (!ign[w * 64 + b]) m |= 1ull << b;
                um[w] = m;
                nun += __popcll(m);
            }
#pragma unroll 1
            for (int i = lane; i < G; i += 32)
                a.o.locus_flags[l0 + l_raw[i]] = WFL_LOCUS_RETAINED | (ign[i] ? WFL_LOCUS_IGNORED : 0);
            nun = warp_sum(nun);
            if (iter == 0 && c == a.dbg_contig) {
#pragma unroll 1
                for (int g = lane; g < Ngrp; g += 32)
                    if (g < a.dbg_cap) {
                        a.dbg_clade[g] = cl_id[g_t[g]];
                        a.dbg_locus[g] = g_loc[g];
                        a.dbg_score[g] = g_score[g];
                    }
                if (lane == 0) *a.dbg_count = Ngrp;
            }
            if (iter == 0 && nun == 0) break;   // "empty" contig, waafle_orgscorer.py:959
            if (a.det_count) {   // write_details (:802-812): the level's gene scores, one entry per (clade, locus) group
                unsigned long long dbase = 0;
                if (lane == 0) dbase = atomicAdd(a.det_count, (unsigned long long)Ngrp);
                dbase = __shfl_sync(FULL, dbase, 0);
#pragma unroll 1
                for (int g = lane; g < Ngrp; g += 32) {
                    const unsigned long long o = dbase + g;
                    if ((long long)o < a.det_cap) {
                        a.det_contig[o] = (int32_t)c;
                        a.det_iter[o] = iter;
                        a.det_clade[o] = cl_id[g_t[g]];
                        a.det_locus[o] = l_raw[g_loc[g]];
                        a.det_score[o] = g_score[g];
                    }
                }
            }
            // ---- clade rows + gene bitmasks ----------------------------------------------------
            // every rank in [0, T) owns >= 1 group (the spiked Unknown owns G)
            DECL_CLADES
            if (!al.ok) { overflow = true; break; }
#pragma unroll 1
            for (int g = lane; g < Ngrp; g += 32)
                if (g == 0 || g_t[g] != g_t[g - 1]) cl_go[g_t[g]] = g;
            if (lane == 0) cl_go[T] = Ngrp;
            hasroot = 0;
#pragma unroll 1
            for (int t = lane; t < T; t += 32) hasroot |= cl_id[t] == tax.root;
            hasroot = __any_sync(FULL, hasroot);
            __syncwarp();
#pragma unroll 1
            for (int t = lane; t < T; t += 32) {
                memA[t] = memB[t] = 0;
                cl_par[t] = tax.listed[cl_id[t]] ? tax.parent[cl_id[t]] : -1;
#pragma unroll 1
                for (int q = 0; q < 3; ++q) {
                    u64 *m = (q == 0 ? mk0 : q == 1 ? mk1 : mk2) + (size_t)t * W;
                    const double thr = q == 0 ? P.p.k1 : q == 1 ? P.p.k2 : 1e-6;
                    // a locus without an entry scores 0 (waafle_orgscorer.py:404-405)
#pragma unroll 1
                    for (int w = 0; w < W; ++w) {
                        int nb = min(64, G - w * 64);
                        m[w] = thr <= 0.0 ? (nb == 64 ? ~0ull : ((1ull << nb) - 1)) : 0ull;
                    }
#pragma unroll 1
                    for (int g = cl_go[t]; g < cl_go[t + 1]; ++g) {
                        int loc = g_loc[g];
                        u64 bit = 1ull << (loc & 63);
                        if (g_score[g] >= thr) m[loc >> 6] |= bit;
                        else m[loc >> 6] &= ~bit;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) *Lp = Level{G, W, T, Ngrp, nun, g_loc, g_score, cl_id, cl_go, {mk0, mk1, mk2}, um, ign, l_len, cl_par};
            __syncwarp();
            cont_ok = true;
        }
        PH_END(4);
        if (overflow) {
            EMIT_RESULT(1);
        } else if (!cont_ok) {
            EMIT_RESULT(0);   // "empty" contig: every locus ignored at the first level (unclassified)
        } else if (lane == 0) {
            PipeCtg *cp = &a.ctg[c];
            cp->nun = nun;
            cp->hasroot = hasroot;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 3: one-clade search
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * WFL_LAT_WPC, WFL_LAT_CPSM) wfl_pipe_one(const PipeArgs a) {
    const int lane = threadIdx.x & 31;
    const DevParams &P = a.P;
    const DevTax &tax = a.t;
    const int S = P.p.n_systems;
#pragma unroll 1
    for (;;) {
        const long long c = pop_work(a.wq, a.list_act, a.cnt_act, lane);
        if (c < 0) break;
        if (a.ctg[c].state != PIPE_ACTIVE) continue;
        PH_BEGIN;
        OPEN_CONTIG
        RESULT_LOCALS
        const int Ngrp = cx.Ngrp, ng = cx.ng;
        DECL_CUR
        DECL_GROUPS
        DECL_CLADES
        (void)cur; (void)s_a; (void)s_b; (void)s_v; (void)g_score; (void)g_rs; (void)g_re; (void)g_loc; (void)g_t; (void)gs; (void)g_perm; (void)gcur;
        (void)cand; (void)memB; (void)mk1; (void)mk2; (void)bestm; (void)cl_go; (void)cl_par;
        const Level &L = *Lp;
        (void)L;
        // ---- K6: one-clade search (explain_one, waafle_orgscorer.py:585-597) -----------
        u64 bbits = 0;
#pragma unroll 1
        for (int t = lane; t < T; t += 32) {
            bool pass = true;
#pragma unroll 1
            for (int w = 0; w < W; ++w) pass &= (mk0[(size_t)t * W + w] & um[w]) == um[w];   // crit >= k1
            cl_opt[t] = pass;
            if (pass) {
                double crit, rank;
                rank = score_clades(Lp, t, -1, &crit);
                cl_rank[t] = rank;
                cl_crit[t] = crit;
                u64 b = dbits(rank);
                bbits = b > bbits ? b : bbits;
            }
        }
        bbits = warp_max_u64(bbits);
        __syncwarp();
        long long bt = -1;
        if (bbits)
            for (int t = lane; t < T; t += 32)
                if (cl_opt[t] && dbits(cl_rank[t]) == bbits) bt = t;   // ties: last in name order
        bt = warp_max_ll(bt);
        if (bt >= 0) {
            {
                // meld_one (waafle_orgscorer.py:621-631)
                const int tb = (int)bt;
                const double brank = cl_rank[tb];
                r_call = WFL_CALL_NO_LGT;
                r_b1 = r_c1 = cl_id[tb];
                r_crit = cl_crit[tb];
                r_rank = brank;
                if (P.p.disambiguate_one == 1) {
                    int my = -1, nk = 0;
#pragma unroll 1
                    for (int t = lane; t < T; t += 32)
                        if (cl_opt[t] && brank - cl_rank[t] <= P.p.range) {
                            my = lca2(tax, my, cl_id[t]);
                            memA[t] = 1;
                            ++nk;
                        }
                    r_c1 = warp_lca(tax, my);
                    r_na = warp_sum(nk);
                }
#pragma unroll 1
                for (int i = lane; i < G; i += 32)   // set_synteny_one (:495-509)
                    a.o.synteny[l0 + l_raw[i]] =
                        ign[i] ? '~' : ((mk0[(size_t)tb * W + (i >> 6)] >> (i & 63)) & 1 ? 'A' : '!');
            }
            if (r_call != WFL_CALL_UNCLASSIFIED) {
                // ---- melded members -> staging pool (tails, waafle_orgscorer.py:630,658-659)
                if (r_na + r_nb > 0) {
                    long long mb = 0;
                    if (lane == 0)
                        mb = (long long)atomicAdd(&a.ctr->mem_pool_used, (unsigned long long)(r_na + r_nb));
                    r_mem = __shfl_sync(FULL, mb, 0);
#pragma unroll 1
                    for (int side = 0; side < 2; ++side) {
                        const u8 *mem = side ? memB : memA;
                        long long off = r_mem + (side ? r_na : 0);
                        if ((side ? r_nb : r_na) == 0) continue;
                        int mbase = 0;
#pragma unroll 1
                        for (int base = 0; base < T; base += 32) {
                            int t = base + lane;
                            bool f = t < T && mem[t];
                            u32 m = __ballot_sync(FULL, f);
                            long long dst = off + mbase + __popc(m & lt_mask());
                            if (f && dst < a.o.mem_pool_cap) a.o.mem_pool[dst] = cl_id[t];
                            mbase += __popc(m);
                        }
                    }
                }
            }
            EMIT_RESULT(0);
        } else if (lane == 0) {
            int slot = atomicAdd(a.cnt_two, 1);
            a.list_two[slot] = (int)c;
        }
        PH_END(5);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 4a: two-clade search and decision; undecided contigs go to the lift list
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32, WFL_PIPE_CPSM) wfl_pipe_two(const PipeArgs a) {
    const int lane = threadIdx.x;
    const DevParams &P = a.P;
    const DevTax &tax = a.t;
    const int S = P.p.n_systems;
    const bool spike = P.p.weak_loci == 2;
#pragma unroll 1
    for (;;) {
        const long long c = pop_work(a.wq, a.list_two, a.cnt_two, lane);
        if (c < 0) break;
        PH_BEGIN;
        OPEN_CONTIG
        RESULT_LOCALS
        const int Ngrp = cx.Ngrp, ng = cx.ng, nu = cx.nu, t_unk = cx.t_unk, hasroot = cx.hasroot;
        DECL_CUR
        DECL_GROUPS
        DECL_CLADES
        (void)cur; (void)s_a; (void)s_b; (void)s_v; (void)g_score; (void)g_rs; (void)g_re; (void)g_loc; (void)g_t; (void)gs; (void)g_perm; (void)gcur;
        (void)cl_rank; (void)cl_crit; (void)cl_opt; (void)mk0; (void)mk2; (void)cl_go; (void)cl_par;
        (void)nu; (void)t_unk; (void)hasroot; (void)spike; (void)T; (void)r_t; (void)r_loc;
        const Level &L = *Lp;
        bool overflow = false, undecided = false;
        long long n_ptest = 0, n_pscore = 0;
#pragma unroll 1
        for (int once = 0; once < 1; ++once) {
            // ---- K7: two-clade search (explain_two, waafle_orgscorer.py:599-619) --------
            int T2 = 0;
#pragma unroll 1
            for (int base = 0; base < T; base += 32) {
                int t = base + lane;
                bool f = false;
                if (t < T)   // max(gene_scores[clade]) >= k2, unmasked (:603-605)
                    for (int w = 0; w < W; ++w) f |= mk1[(size_t)t * W + w] != 0;
                u32 m = __ballot_sync(FULL, f);
                if (f) cand[T2 + __popc(m & lt_mask())] = t;
                T2 += __popc(m);
            }
            __syncwarp();
            const long long NP = (long long)T2 * (T2 - 1) / 2;
            n_ptest += NP;
            // pass 1: mask prefilter over all pairs (crit >= k2 <=> every non-ignored locus is
            // covered at k2 by one of the two clades); survivors are compacted in pair order
            size_t room = al.cap > al.used ? al.cap - al.used : 0;
            long long scap = ((long long)room - 4LL * (T + 1) - 8LL * (BITMAP_MAX_WORDS >= ((tax.n_nodes + 31) >> 5) ? ((tax.n_nodes + 31) >> 5) : 0) - 512) / 16;   // leave room for the lift's tables
            if (scap > NP) scap = NP;
            if (scap < 0) scap = 0;
            LinArena ax = al;
            if (scap < NP) {   // not one slot per pair: take a fresh piece of the workspace pool
                const unsigned long long want = 16ull * (unsigned long long)NP + 256ull;
                unsigned long long off = 0;
                if (lane == 0) off = atomicAdd(a.pool_used, (want + 255ull) & ~255ull);
                off = __shfl_sync(FULL, off, 0);
                if (off + want <= a.pool_cap) {
                    ax = LinArena{a.pool + off, (size_t)want, 0, true};
                    scap = NP;
                }
            }
            int *s_i = ax.get<int>((size_t)scap), *s_j = ax.get<int>((size_t)scap);
            double *s_rank = ax.get<double>((size_t)scap);
            if (!ax.ok) { overflow = true; break; }
            if (!al.ok) { overflow = true; break; }
            int nsurv = 0;
            {
                int pi = 0, po = 0;   // lane's pair: clade cand[pi] with cand[pi + 1 + po]
                if (lane < NP) {
                    int jj;
                    pair_decode(lane, T2, pi, jj);
                    po = jj - pi - 1;
                }
#pragma unroll 1
                for (long long pb = 0; pb < NP; pb += 32) {
                    const bool act = pb + lane < NP;
                    bool pass = false;
                    if (act) pass = pair_pass(L, cand[pi], cand[pi + 1 + po]);   // crit < k2 fails (:610)
                    u32 m = __ballot_sync(FULL, pass);
                    if (pass) {
                        long long dst = (long long)nsurv + __popc(m & lt_mask());
                        if (dst < scap) { s_i[dst] = pi; s_j[dst] = pi + 1 + po; }
                    }
                    nsurv += __popc(m);
                    if (act) {   // advance the lane's pair by 32 in i-major order
                        po += 32;
                        while (pi < T2 - 1 && po >= T2 - 1 - pi) { po -= T2 - 1 - pi; ++pi; }
                    }
                }
            }
            if (nsurv > scap) {   // survivor list does not fit: replay with a slab sized for all pairs
                overflow = true;
                break;
            }
            n_pscore += nsurv;
            __syncwarp();
            // pass 2: exact crit / rank of the survivors; best rank, ties -> last pair in
            // (clade1, clade2) iteration order
            double my_rank = -1.0;
            long long my_p = -1;
#pragma unroll 1
            for (int q = lane; q < nsurv; q += 32) {
                double crit;
                double rank = score_clades(Lp, cand[s_i[q]], cand[s_j[q]], &crit);
                s_rank[q] = rank;
                if (my_p < 0 || rank >= my_rank) { my_rank = rank; my_p = q; }
            }
            u64 pb = warp_max_u64(my_p >= 0 ? dbits(my_rank) : 0ull);
            const long long bp = warp_max_ll((my_p >= 0 && dbits(my_rank) == pb) ? my_p : -1);
            __syncwarp();
            if (bp >= 0) {
                // meld_two (waafle_orgscorer.py:633-669)
                const int bi = s_i[bp], bj = s_j[bp];
                TwoEval be;
                eval_two(L, tax, P, cand[bi], cand[bj], be);
                double bcrit, brank;
                brank = score_clades(Lp, cand[bi], cand[bj], &bcrit);
                const bool bunk = be.c1 == tax.unknown || be.c2 == tax.unknown;
#pragma unroll 1
                for (int w = lane; w < W; w += 32) {
                    u64 A, Bm, amb;
                    letters(L, L.mk[P.amb_sel], bunk, cand[bi], cand[bj], w, A, Bm, amb);
                    bestm[w] = be.swap ? Bm : A;
                    bestm[W + w] = be.swap ? A : Bm;
                    bestm[2 * W + w] = amb;
                }
                __syncwarp();
                int nk = 0, nbad = 0, ndiff = 0, la = -1, lb = -1;
#pragma unroll 1
                for (int q = lane; q < nsurv; q += 32) {
                    if (!(brank - s_rank[q] <= P.p.range)) continue;   // :636
                    const int t1 = cand[s_i[q]], t2 = cand[s_j[q]];
                    TwoEval ev;
                    eval_two(L, tax, P, t1, t2, ev);
                    ++nk;
                    nbad += !ev.ok;
                    const bool unk = ev.c1 == tax.unknown || ev.c2 == tax.unknown;
                    bool same = true;   // meld_precheck: same synteny string (:671-676)
#pragma unroll 1
                    for (int w = 0; w < W; ++w) {
                        u64 A, Bm, amb;
                        letters(L, L.mk[P.amb_sel], unk, t1, t2, w, A, Bm, amb);
                        same &= (ev.swap ? Bm : A) == bestm[w] && (ev.swap ? A : Bm) == bestm[W + w] &&
                                amb == bestm[2 * W + w];
                    }
                    ndiff += !same;
                    la = lca2(tax, la, ev.c1);
                    lb = lca2(tax, lb, ev.c2);
                    memA[ev.t1] = 1;
                    memB[ev.t2] = 1;
                }
                nk = warp_sum(nk);
                nbad = warp_sum(nbad);
                ndiff = warp_sum(ndiff);
                la = warp_lca(tax, la);
                lb = warp_lca(tax, lb);
                __syncwarp();
                bool have = true, melded = false;
                int c1 = be.c1, c2 = be.c2;
                if (nk == 1 || P.p.disambiguate_two == 0) {
                } else if (P.p.disambiguate_two == 1) {
                    have = false;
                } else if (nbad > 0 || ndiff > 0) {
                    have = false;
                } else {
                    c1 = la;
                    c2 = lb;
                    melded = true;
                    if (!P.p.allow_lca) {   // post-meld LCA check (:661-665)
                        int l = lca2(tax, c1, c2);
                        if (l == c1 || l == c2) have = false;
                    }
                }
                if (have && be.ok) {
                    r_call = WFL_CALL_LGT;
                    r_b1 = be.c1;
                    r_b2 = be.c2;
                    r_c1 = c1;
                    r_c2 = c2;
                    r_lca = lca2(tax, c1, c2);   // waafle_orgscorer.py:882
                    r_crit = bcrit;
                    r_rank = brank;
                    r_dir = be.dir;
                    if (melded) {
                        int na = 0, nb = 0;
#pragma unroll 1
                        for (int t = lane; t < T; t += 32) { na += memA[t]; nb += memB[t]; }
                        r_na = warp_sum(na);
                        r_nb = warp_sum(nb);
                    }
#pragma unroll 1
                    for (int i = lane; i < G; i += 32) {
                        u64 m = 1ull << (i & 63);
                        int w = i >> 6;
                        a.o.synteny[l0 + l_raw[i]] = ign[i] ? '~' : (bestm[2 * W + w] & m) ? '*'
                                                     : (bestm[w] & m) ? 'A' : (bestm[W + w] & m) ? 'B' : '!';
                    }
                }
            }
            if (r_call != WFL_CALL_UNCLASSIFIED) {
                // ---- melded members -> staging pool (tails, waafle_orgscorer.py:630,658-659)
                if (r_na + r_nb > 0) {
                    long long mb = 0;
                    if (lane == 0)
                        mb = (long long)atomicAdd(&a.ctr->mem_pool_used, (unsigned long long)(r_na + r_nb));
                    r_mem = __shfl_sync(FULL, mb, 0);
#pragma unroll 1
                    for (int side = 0; side < 2; ++side) {
                        const u8 *mem = side ? memB : memA;
                        long long off = r_mem + (side ? r_na : 0);
                        if ((side ? r_nb : r_na) == 0) continue;
                        int mbase = 0;
#pragma unroll 1
                        for (int base = 0; base < T; base += 32) {
                            int t = base + lane;
                            bool f = t < T && mem[t];
                            u32 m = __ballot_sync(FULL, f);
                            long long dst = off + mbase + __popc(m & lt_mask());
                            if (f && dst < a.o.mem_pool_cap) a.o.mem_pool[dst] = cl_id[t];
                            mbase += __popc(m);
                        }
                    }
                }
                break;
            }
            undecided = true;
        }
        if (lane == 0) {
            if (n_ptest) atomicAdd(&a.ctr->pairs_tested, (unsigned long long)n_ptest);
            if (n_pscore) atomicAdd(&a.ctr->pairs_scored, (unsigned long long)n_pscore);
        }
        if (overflow) {
            r_call = WFL_CALL_UNCLASSIFIED;
            r_na = r_nb = 0;
            EMIT_RESULT(1);
        } else if (!undecided) {
            EMIT_RESULT(r_status);
        } else if (lane == 0) {
            int slot = atomicAdd(a.cnt_lift, 1);
            a.list_lift[slot] = (int)c;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 4b: stop (root reached / nothing left) or lift the clade table to the parents (K9, K5)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * WFL_LAT_WPC, WFL_LAT_CPSM) wfl_pipe_lift(const PipeArgs a) {
    const int lane = threadIdx.x & 31;
    const DevParams &P = a.P;
    const DevTax &tax = a.t;
    const int S = P.p.n_systems;
    const bool spike = P.p.weak_loci == 2;
#pragma unroll 1
    for (;;) {
        const long long c = pop_work(a.wq, a.list_lift, a.cnt_lift, lane);
        if (c < 0) break;
        PH_BEGIN;
        OPEN_CONTIG
        RESULT_LOCALS
        const int Ngrp = cx.Ngrp, ng = cx.ng, nu = cx.nu, t_unk = cx.t_unk, hasroot = cx.hasroot;
        DECL_CUR
        DECL_GROUPS
        DECL_CLADES
        (void)cur; (void)s_a; (void)s_b; (void)s_v; (void)g_score; (void)g_rs; (void)g_re; (void)g_loc; (void)g_t; (void)gs; (void)g_perm; (void)gcur;
        (void)cl_rank; (void)cl_crit; (void)cl_opt; (void)mk0; (void)mk1; (void)mk2; (void)cl_go; (void)cl_par; (void)cand;
        (void)memA; (void)memB; (void)bestm; (void)Lp; (void)nu; (void)t_unk; (void)r_loc; (void)l_raw; (void)l0; (void)ign; (void)um;
        bool overflow = false, lifted = false;
#pragma unroll 1
        for (int once = 0; once < 1; ++once) {
            // not explained at this level: stop or lift (waafle_orgscorer.py:571-575)
            if (T == 0 || hasroot) break;
            if (iter >= 100) { r_status = 2; break; }   // :580-581
            // ---- K5: lift the distinct-clade table (raise_taxonomy, :431-445) ----------------
            // parents of the T clades, deduped and re-ranked (rank by counting); records follow
            // through map_t.  "Unknown" spiked at this level is not a site-score clade: it is
            // dropped here and re-inserted (:418, :433-443).
            {
                int *par = al.get<int>(T + 1);
                if (!al.ok) { overflow = true; break; }
                bool rec_unknown = false;   // does a record clade equal Unknown? (hit taxon named so)
                if (spike) rec_unknown = nu > 0;
#pragma unroll 1
                for (int t = lane; t < T; t += 32) {
                    bool drop = spike && t == t_unk && !rec_unknown;
                    par[t] = drop ? -1 : tax.parent[cl_id[t]];
                }
                if (lane == 0) par[T] = spike ? tax.unknown : -1;   // re-inserted spike key
                __syncwarp();
                int Tn = 0;
                const int nwl = (tax.n_nodes + 31) >> 5;
                if (nwl <= BITMAP_MAX_WORDS) {
                    // small taxonomies: presence bitmap of the parents, new rank = prefix popcount
                    u32 *bm = al.get<u32>(nwl);
                    int *bpre = al.get<int>(nwl + 1);
                    if (!al.ok) { overflow = true; break; }
#pragma unroll 1
                    for (int w = lane; w < nwl; w += 32) bm[w] = 0;
                    __syncwarp();
#pragma unroll 1
                    for (int t = lane; t <= T; t += 32)
                        if (par[t] >= 0) atomicOr(&bm[par[t] >> 5], 1u << (par[t] & 31));
                    __syncwarp();
#pragma unroll 1
                    for (int base = 0; base < nwl; base += 32) {
                        const int w = base + lane;
                        int tot, ex = warp_excl_scan(w < nwl ? __popc(bm[w]) : 0, tot);
                        if (w < nwl) bpre[w] = Tn + ex;
                        Tn += tot;
                    }
                    __syncwarp();
#pragma unroll 1
                    for (int t = lane; t <= T; t += 32) {
                        const int key = par[t];
                        map_t[t] = key < 0 ? -1 : bpre[key >> 5] + __popc(bm[key >> 5] & ((1u << (key & 31)) - 1u));
                    }
                } else {
#pragma unroll 1
                for (int base = 0; base <= T; base += 32) {   // first occurrences of each key
                    int t = base + lane;
                    bool f = false;
                    if (t <= T && par[t] >= 0) {
                        f = true;
#pragma unroll 1
                        for (int z = 0; z < t; ++z)
                            if (par[z] == par[t]) { f = false; break; }
                    }
                    if (t <= T) fo[t] = f;
                    Tn += __popc(__ballot_sync(FULL, f));
                }
                __syncwarp();
#pragma unroll 1
                for (int t = lane; t <= T; t += 32) {   // rank = #distinct keys below
                    int key = par[t], rk = -1;
                    if (key >= 0) {
                        rk = 0;
#pragma unroll 1
                        for (int q = 0; q <= T; ++q) rk += fo[q] && par[q] < key;
                    }
                    map_t[t] = rk;
                }
                }
                __syncwarp();
#pragma unroll 1
                for (int r = lane; r < M; r += 32) r_t[r] = map_t[r_t[r]];
                __syncwarp();
#pragma unroll 1
                for (int t = lane; t <= T; t += 32)
                    if (map_t[t] >= 0) cl_id[map_t[t]] = par[t];   // equal keys write equal values
                T = Tn;
                __syncwarp();
            }
            ++lifts;
            lifted = true;
        }
        PH_END(7);
        if (overflow) {
            r_call = WFL_CALL_UNCLASSIFIED;
            r_na = r_nb = 0;
            EMIT_RESULT(1);
        } else if (!lifted) {
            EMIT_RESULT(r_status);
        } else if (lane == 0) {
            PipeCtg *cp = &a.ctg[c];
            cp->T = T;
            cp->lifts = lifts;
            cp->iter = iter + 1;
            int slot = atomicAdd(a.cnt_next, 1);
            a.list_next[slot] = (int)c;
        }
        __syncwarp();
    }
}

// Contigs still on the work list after the last level: every lift moves the shallowest clade one level up, so
// max depth + 1 levels always suffice -- anything left is runaway recursion (waafle_orgscorer.py:580-581).
__global__ void wfl_pipe_leftover(const PipeArgs a) {
    const int n = *a.cnt_act;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int c = a.list_act[i];
        a.o.status[c] = 2;
        a.o.call[c] = WFL_CALL_UNCLASSIFIED;
        a.o.n_mem_a[c] = a.o.n_mem_b[c] = 0;
        atomicAdd(&a.ctr->n_runaway, 1ull);
    }
}

// ---------------------------------------------------------------------------------------------
// host side: launch sequence for one sub-batch
// ---------------------------------------------------------------------------------------------
void launch_pipe_prepare(const PipeArgs &a, int grid, cudaStream_t s) { wfl_pipe_prepare<<<grid, 32, 0, s>>>(a); }
void launch_pipe_regroup(const PipeArgs &a, int grid, cudaStream_t s) { wfl_pipe_regroup<<<grid / WFL_PIPE_CPSM * WFL_LAT_CPSM, 32 * WFL_LAT_WPC, 0, s>>>(a); }
void launch_pipe_k2sort(const PipeArgs &a, int grid, cudaStream_t s) {
    wfl_pipe_k2hist<<<grid / 8 + 1, 256, 0, s>>>(a);
    wfl_pipe_k2scan<<<1, K2_KEYS, 0, s>>>(a);
    wfl_pipe_k2scatter<<<grid / 8 + 1, 256, 0, s>>>(a);
}
void launch_pipe_k2(const PipeArgs &a, int grid, cudaStream_t s) { wfl_pipe_k2<<<grid, 32, 0, s>>>(a); }
void launch_pipe_masks(const PipeArgs &a, int grid, cudaStream_t s) { wfl_pipe_masks<<<grid / WFL_PIPE_CPSM * WFL_LAT_CPSM, 32 * WFL_LAT_WPC, 0, s>>>(a); }
void launch_pipe_one(const PipeArgs &a, int grid, cudaStream_t s) { wfl_pipe_one<<<grid / WFL_PIPE_CPSM * WFL_LAT_CPSM, 32 * WFL_LAT_WPC, 0, s>>>(a); }
void launch_pipe_two(const PipeArgs &a, int grid, cudaStream_t s) { wfl_pipe_two<<<grid, 32, 0, s>>>(a); }
void launch_pipe_lift(const PipeArgs &a, int grid, cudaStream_t s) { wfl_pipe_lift<<<grid / WFL_PIPE_CPSM * WFL_LAT_CPSM, 32 * WFL_LAT_WPC, 0, s>>>(a); }
int pipe_ctas_per_sm() { return WFL_PIPE_CPSM; }
void launch_pipe_leftover(const PipeArgs &a, cudaStream_t s) { wfl_pipe_leftover<<<64, 256, 0, s>>>(a); }

}  // namespace wfl
