// The wide scoring batch (wfl_batch) built on the device from the hit columns a wfl_parser keeps there, with the bytes
// packing.pack(...) produces on the host: contig c of the batch takes the parser rows of its blastout block, the taxon
// slot becomes the node index through the caller's table, the raw system bits become the sorted system bits
// (wfl_parse_sysmask's rule), and without annotation systems every contig's hits are put in Batch.sort_hits order.
//
//   wfl_resident_gather  one thread per batch hit: validates the taxon slot, reduces the largest finite score > 0 and
//                        the largest node (sort_hits' smax and bits_t), and copies the row when no sort follows;
//   wfl_resident_sort    one warp per contig: builds the contig's 128-bit keys in a scratch slice, sorts them with the
//                        bitonic network of the details table (wfl_warp_sort.cuh) and writes the rows in key order.
//                        Contigs whose keys exceed the first launch's slice go to a second launch sized for the largest.
#include <algorithm>

#include "wfl_warp_sort.cuh"

namespace wfl {
namespace {

// contig of batch hit h: the last c with hit_off[c] <= h (contigs without hits are skipped over)
__device__ __forceinline__ long long contig_of(const int64_t *hit_off, long long n, long long h) {
    long long lo = 0, hi = n - 1;
    while (lo < hi) {
        const long long mid = (lo + hi + 1) >> 1;
        if (hit_off[mid] <= h) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ int node_of(const ResBatchArgs &a, long long row) {
    const int slot = a.tcode[row];
    return (unsigned)slot < (unsigned)a.n_slots ? a.slot_node[slot] : -1;
}

__device__ __forceinline__ void put_hit(const ResBatchArgs &a, long long h, long long row, int node) {
    a.o_qstart[h] = a.qstart[row];
    a.o_qend[h] = a.qend[row];
    a.o_taxon[h] = node;
    a.o_score[h] = a.score[row];
    a.o_scov[h] = a.scov[row];
    a.o_strand[h] = a.strand[row];
    if (a.sys_perm) {
        u64 m = a.rawmask[row];
        u32 out = 0;
        while (m) {
            const int b = __ffsll((long long)m) - 1;
            m &= m - 1;
            if (a.sys_perm[b] >= 0) out |= 1u << a.sys_perm[b];
        }
        a.o_sysmask[h] = out;
    }
}

__global__ void __launch_bounds__(256) wfl_resident_gather(const ResBatchArgs a) {
    u64 bad = 0, smax = 0, tmax = 0;
    for (long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x; h < a.nh; h += (long long)gridDim.x * blockDim.x) {
        const long long c = contig_of(a.hit_off, a.n, h);
        const long long row = a.hit_src[c] + (h - a.hit_off[c]);
        const int node = node_of(a, row);
        if (node < 0 || node >= a.n_nodes) { ++bad; continue; }
        tmax = max(tmax, (u64)node);
        const double s = a.score[row];
        // np.nan_to_num maps NaN and +-inf to 0, and the max starts at 0: only finite s > 0 count.  Positive doubles
        // order like their bit patterns.
        if (s > 0.0 && s <= 1.7976931348623157e308) smax = max(smax, (u64)__double_as_longlong(s));
        if (a.sys_perm) put_hit(a, h, row, node);   // with annotation systems the hits stay in file order
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(FULL, bad, o);
        smax = max(smax, (u64)__shfl_xor_sync(FULL, smax, o));
        tmax = max(tmax, (u64)__shfl_xor_sync(FULL, tmax, o));
    }
    if (lane_id() == 0) {
        if (bad) atomicAdd(&a.red[0], bad);
        if (smax) atomicMax(&a.red[1], smax);
        if (tmax) atomicMax(&a.red[2], tmax);
    }
}

__global__ void __launch_bounds__(256) wfl_resident_sort(const ResBatchArgs a) {
    const int lane = lane_id();
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    ulonglong2 *v = reinterpret_cast<ulonglong2 *>(a.scratch + warp * a.slice);
    // the quantisation of sort_hits: q = (int64)((smax - clip(s, 0, smax)) * (float((1 << bits_s) - 1) / smax)), rounded
    // step by step as numpy rounds it (no fused multiply-add)
    const double scale = a.quantised ? __ddiv_rn((double)((1ll << a.bits_s) - 1), a.smax) : 0.0;
    const long long n_work = a.list ? a.n_list : a.n;
    for (long long w = warp; w < n_work; w += nwarps) {
        const long long c = a.list ? a.list[w] : w;
        const long long h0 = a.hit_off[c], src = a.hit_src[c];
        const int H = (int)(a.hit_off[c + 1] - h0);
        const int NP = pow2_at_least(H);
        if (H == 0 || (!a.list && 16ll * NP > a.slice)) continue;   // the big ones are the second launch's
        for (int i = lane; i < NP; i += 32) {
            ulonglong2 k = make_ulonglong2(~0ull, ~0ull);
            if (i < H) {
                const long long row = src + i;
                const u64 node = (u64)node_of(a, row);
                const double s = a.score[row];
                if (a.quantised) {
                    const double sf = (s == s && s - s == 0.0) ? s : 0.0;   // nan_to_num
                    const double cl = fmin(fmax(sf, 0.0), a.smax);
                    const long long q = (long long)__dmul_rn(__dsub_rn(a.smax, cl), scale);
                    k = make_ulonglong2((node << a.bits_s) | (u64)q, (u64)i);
                } else {
                    // np.lexsort((row, -score, taxon)): -0.0 ties with +0.0 (dbits), NaN sorts last
                    const double ns = -s;
                    const u64 kb = ns == ns ? dbits(ns) : ~0ull;
                    k = make_ulonglong2((node << 32) | (kb >> 32), (kb << 32) | (u64)i);
                }
            }
            v[i] = k;
        }
        __syncwarp();
        warp_sort(v, NP);
        for (int j = lane; j < H; j += 32) {
            const long long row = src + (long long)(u32)v[j].y;
            put_hit(a, h0 + j, row, node_of(a, row));
        }
        __syncwarp();
    }
}

}  // namespace

void launch_resident_gather(const ResBatchArgs &a, int sm_count, cudaStream_t s) {
    const long long blocks = std::min<long long>((a.nh + 255) / 256, (long long)sm_count * 16);
    wfl_resident_gather<<<(int)std::max<long long>(1, blocks), 256, 0, s>>>(a);
}

void launch_resident_sort(const ResBatchArgs &a, long long warps, cudaStream_t s) {
    wfl_resident_sort<<<(int)std::max<long long>(1, (warps + 7) / 8), 256, 0, s>>>(a);
}

}  // namespace wfl
