// BGZF blastouts inflated on the device (SURVEY 8f f1): the compressed bytes cross PCIe, the text is written straight
// into the parser's resident text buffer, and wfl_parse_blast_resident parses it where it lies.
//
// BGZF (the gzip variant bgzip writes) is a series of independent gzip members of <= 64 KB of text each; every member's
// header holds its compressed size and its trailer its text size (ISIZE) and CRC-32, so the host knows every member's
// payload and output offset before anything is decoded (waafle_b200/compressed.py builds that member table).
//
//   wfl_inflate_members   one thread per member: the member's DEFLATE stream (RFC 1951: stored, fixed- and
//                         dynamic-Huffman blocks, any number of them) is decoded serially into its slice of the text,
//                         then its CRC-32 is compared with the trailer's.  A member that fails any check marks the file
//                         (atomicMin of its index); the caller then reads the file on the host, which raises the error
//                         Python's gzip raises.
//
// Why one thread per member: DEFLATE decoding is serial inside a member, and a blastout of any size worth inflating on
// the device has tens of thousands of members (2.5 GB of text = 40 000), which is the parallelism.  The decoder is one
// __host__ __device__ function (the INFLATE-HOST region below), so the host build that tests it against zlib, corrupt
// inputs and the address sanitizer (tests/test_compressed.py) runs exactly the code the kernel runs.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>

#include "waafle_b200.h"
#include "wfl_parser.cuh"

#define WFL_HD __host__ __device__

namespace wfl {

// INFLATE-HOST-BEGIN
// ---- one DEFLATE stream with every input checked (the file comes from outside the program) -------------------------
// Errors: the bit reader never reads past the payload, over-subscribed code-length sets and incomplete ones (except a
// single code of one bit, and an empty distance code, as zlib allows) are rejected, literal/length symbols 286-287 and
// distance codes 30-31 are rejected, no match reaches before the start of the member's output (BGZF members share no
// window), the output must be exactly ISIZE bytes, the stream must end exactly at the end of the payload, and the CRC-32
// must match the trailer.
enum {
    INF_OK = 0,
    INF_E_TRUNC = -1,     // the payload ended inside the stream
    INF_E_BTYPE = -2,     // block type 3
    INF_E_STORED = -3,    // stored block: LEN != ~NLEN
    INF_E_CODES = -4,     // bad code-length set (over-subscribed, incomplete, bad repeat, no end-of-block code)
    INF_E_SYMBOL = -5,    // a code not in the table, literal/length 286-287, distance 30-31
    INF_E_DIST = -6,      // a distance before the start of the member's output
    INF_E_SIZE = -7,      // output past ISIZE or short of it
    INF_E_TRAIL = -8,     // bytes left over between the end of the stream and the end of the payload
    INF_E_CRC = -9,       // CRC-32 differs from the trailer's
};

constexpr int INF_FAST = 10;   // codes of <= 10 bits decode with one table lookup

struct InfHuff {
    uint16_t fast[1 << INF_FAST];   // (code length << 9) | symbol, indexed by the next INF_FAST bits; 0 = longer code / none
    uint16_t count[16];             // codes per length
    uint16_t sym[288];              // symbols ordered by (length, symbol): the canonical order
};

struct InfState {
    const uint8_t *in;
    uint32_t n, pos;   // payload bytes, next byte to load
    uint64_t buf;      // bit buffer (LSB first)
    int cnt;           // bits in buf
    uint8_t *out;
    uint32_t olen, op;
};

// Canonical Huffman table of n code lengths.  Returns the unused code space (0 = complete, > 0 incomplete) or -1 when
// the set is over-subscribed.
WFL_HD inline int inf_build(InfHuff &h, const uint8_t *len, int n) {
    for (int l = 0; l < 16; ++l) h.count[l] = 0;
    for (int s = 0; s < n; ++s) h.count[len[s]]++;
    int left = 1;
    for (int l = 1; l < 16; ++l) {
        left <<= 1;
        left -= h.count[l];
        if (left < 0) return -1;
    }
    uint16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + h.count[l];
    for (int s = 0; s < n; ++s)
        if (len[s]) h.sym[offs[len[s]]++] = (uint16_t)s;
    for (int i = 0; i < (1 << INF_FAST); ++i) h.fast[i] = 0;
    unsigned code = 0;
    int idx = 0;
    for (int l = 1; l <= INF_FAST; ++l) {
        for (int k = 0; k < h.count[l]; ++k, ++code, ++idx) {
            unsigned r = 0;   // Huffman codes are sent most significant bit first
            for (int b = 0; b < l; ++b) r |= ((code >> b) & 1u) << (l - 1 - b);
            for (unsigned j = r; j < (1u << INF_FAST); j += 1u << l) h.fast[j] = (uint16_t)((l << 9) | h.sym[idx]);
        }
        code <<= 1;
    }
    return left;
}

WFL_HD inline void inf_fill(InfState &s) {
    while (s.cnt <= 56 && s.pos < s.n) {
        s.buf |= (uint64_t)s.in[s.pos++] << s.cnt;
        s.cnt += 8;
    }
}

WFL_HD inline int inf_bits(InfState &s, int k, uint32_t &v) {   // k <= 32
    if (s.cnt < k) {
        inf_fill(s);
        if (s.cnt < k) return INF_E_TRUNC;
    }
    v = (uint32_t)(s.buf & ((1ull << k) - 1));
    s.buf >>= k;
    s.cnt -= k;
    return INF_OK;
}

// next symbol of table h, or a negative INF_E_*
WFL_HD inline int inf_decode(InfState &s, const InfHuff &h) {
    if (s.cnt < 15) inf_fill(s);
    const unsigned e = h.fast[s.buf & ((1u << INF_FAST) - 1)];
    if (e) {
        const int l = (int)(e >> 9);
        if (l > s.cnt) return INF_E_TRUNC;   // the code's bits run past the payload (the rest of the index was zero fill)
        s.buf >>= l;
        s.cnt -= l;
        return (int)(e & 511u);
    }
    int code = 0, first = 0, index = 0;   // longer codes: walk the canonical code bit by bit
    for (int l = 1; l < 16; ++l) {
        if (l > s.cnt) return INF_E_TRUNC;
        code |= (int)((s.buf >> (l - 1)) & 1u);
        const int c = h.count[l];
        if (code - c < first) {
            s.buf >>= l;
            s.cnt -= l;
            return h.sym[index + (code - first)];
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return INF_E_SYMBOL;   // bits that are no code of an incomplete set
}

// literal/length and distance codes of one block until its end-of-block symbol
WFL_HD inline int inf_codes(InfState &s, const InfHuff &lc, const InfHuff &dc) {
    for (;;) {
        int sym = inf_decode(s, lc);
        if (sym < 0) return sym;
        if (sym < 256) {
            if (s.op >= s.olen) return INF_E_SIZE;
            s.out[s.op++] = (uint8_t)sym;
            continue;
        }
        if (sym == 256) return INF_OK;
        sym -= 257;
        if (sym >= 29) return INF_E_SYMBOL;
        uint32_t len, x;
        if (sym < 8) {
            len = 3 + sym;
        } else if (sym == 28) {
            len = 258;
        } else {
            const int ext = (sym - 4) >> 2;
            if (inf_bits(s, ext, x)) return INF_E_TRUNC;
            len = ((4u + (sym & 3)) << ext) + 3 + x;
        }
        const int d = inf_decode(s, dc);
        if (d < 0) return d;
        if (d >= 30) return INF_E_SYMBOL;
        uint32_t dist;
        if (d < 4) {
            dist = d + 1;
        } else {
            const int ext = (d - 2) >> 1;
            if (inf_bits(s, ext, x)) return INF_E_TRUNC;
            dist = ((2u + (d & 1)) << ext) + 1 + x;
        }
        if (dist > s.op) return INF_E_DIST;
        if (len > s.olen - s.op) return INF_E_SIZE;
        uint8_t *o = s.out + s.op;
        const uint8_t *f = o - dist;
        for (uint32_t i = 0; i < len; ++i) o[i] = f[i];   // in order: an overlapping match repeats its own output
        s.op += len;
    }
}

// A set of code lengths zlib accepts although it is incomplete: one code of one bit (or, for distances, none at all).
WFL_HD inline bool inf_complete_enough(const InfHuff &h, int left, bool may_be_empty) {
    if (left == 0) return true;
    int used = 0;
    for (int l = 1; l < 16; ++l) used += h.count[l];
    return (used == 1 && h.count[1] == 1) || (may_be_empty && used == 0);
}

WFL_HD inline int inf_dynamic(InfState &s, InfHuff &lc, InfHuff &dc, uint8_t *lens) {
    uint32_t nlen, ndist, ncode, v;
    if (inf_bits(s, 5, nlen) || inf_bits(s, 5, ndist) || inf_bits(s, 4, ncode)) return INF_E_TRUNC;
    nlen += 257;
    ndist += 1;
    ncode += 4;
    if (nlen > 286 || ndist > 30) return INF_E_CODES;
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    for (int i = 0; i < 19; ++i) lens[i] = 0;
    for (uint32_t i = 0; i < ncode; ++i) {
        if (inf_bits(s, 3, v)) return INF_E_TRUNC;
        lens[order[i]] = (uint8_t)v;
    }
    if (inf_build(dc, lens, 19) != 0) return INF_E_CODES;   // the code-length code must be complete (dc is scratch here)
    uint32_t i = 0;
    while (i < nlen + ndist) {
        const int sym = inf_decode(s, dc);
        if (sym < 0) return sym;
        if (sym < 16) {
            lens[i++] = (uint8_t)sym;
            continue;
        }
        uint8_t val = 0;
        uint32_t rep;
        if (sym == 16) {
            if (i == 0) return INF_E_CODES;   // repeat without a previous length
            val = lens[i - 1];
            if (inf_bits(s, 2, rep)) return INF_E_TRUNC;
            rep += 3;
        } else if (sym == 17) {
            if (inf_bits(s, 3, rep)) return INF_E_TRUNC;
            rep += 3;
        } else {
            if (inf_bits(s, 7, rep)) return INF_E_TRUNC;
            rep += 11;
        }
        if (i + rep > nlen + ndist) return INF_E_CODES;
        while (rep--) lens[i++] = val;
    }
    if (lens[256] == 0) return INF_E_CODES;   // no end-of-block code
    int left = inf_build(lc, lens, (int)nlen);
    if (left < 0 || !inf_complete_enough(lc, left, false)) return INF_E_CODES;
    left = inf_build(dc, lens + nlen, (int)ndist);
    if (left < 0 || !inf_complete_enough(dc, left, true)) return INF_E_CODES;
    return inf_codes(s, lc, dc);
}

WFL_HD inline int inf_fixed(InfState &s, InfHuff &lc, InfHuff &dc, uint8_t *lens) {
    for (int i = 0; i < 288; ++i) lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
    inf_build(lc, lens, 288);
    for (int i = 0; i < 32; ++i) lens[i] = 5;
    inf_build(dc, lens, 32);   // codes 30-31 exist in the fixed code and are rejected when they occur
    return inf_codes(s, lc, dc);
}

WFL_HD inline int inf_stored(InfState &s) {
    s.buf >>= (s.cnt & 7);   // to the byte boundary
    s.cnt &= ~7;
    uint32_t len, nlen, v;
    if (inf_bits(s, 16, len) || inf_bits(s, 16, nlen)) return INF_E_TRUNC;
    if (len != (~nlen & 0xffffu)) return INF_E_STORED;
    if (len > s.olen - s.op) return INF_E_SIZE;
    for (uint32_t i = 0; i < len; ++i) {
        if (inf_bits(s, 8, v)) return INF_E_TRUNC;
        s.out[s.op++] = (uint8_t)v;
    }
    return INF_OK;
}

// CRC-32 (zlib's polynomial) by 4 bytes at a time: t = 4 x 256 entries from inf_crc_tables
WFL_HD inline void inf_crc_tables(uint32_t *t) {
    for (uint32_t n = 0; n < 256; ++n) {
        uint32_t c = n;
        for (int k = 0; k < 8; ++k) c = c & 1 ? 0xedb88320u ^ (c >> 1) : c >> 1;
        t[n] = c;
    }
    for (int j = 1; j < 4; ++j)
        for (uint32_t n = 0; n < 256; ++n) t[256 * j + n] = (t[256 * (j - 1) + n] >> 8) ^ t[t[256 * (j - 1) + n] & 255];
}

WFL_HD inline uint32_t inf_crc32(const uint32_t *t, const uint8_t *p, uint32_t n) {
    uint32_t c = 0xffffffffu;
    for (; n >= 4; n -= 4, p += 4) {
        c ^= (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
        c = t[768 + (c & 255)] ^ t[512 + ((c >> 8) & 255)] ^ t[256 + ((c >> 16) & 255)] ^ t[c >> 24];
    }
    for (; n; --n) c = t[(c ^ *p++) & 255] ^ (c >> 8);
    return ~c;
}

// One BGZF member: the raw DEFLATE payload in[0, n) -> out[0, isize), checked against the trailer's ISIZE and CRC-32.
// lc / dc / lens (>= 320 bytes) are the caller's scratch.  Returns INF_OK or an INF_E_* code.
WFL_HD inline int inf_member(const uint8_t *in, uint32_t n, uint8_t *out, uint32_t isize, uint32_t crc,
                             const uint32_t *crc_t, InfHuff &lc, InfHuff &dc, uint8_t *lens) {
    InfState s;
    s.in = in; s.n = n; s.pos = 0; s.buf = 0; s.cnt = 0;
    s.out = out; s.olen = isize; s.op = 0;
    uint32_t last, type;
    do {
        if (inf_bits(s, 1, last) || inf_bits(s, 2, type)) return INF_E_TRUNC;
        int rc;
        if (type == 0) rc = inf_stored(s);
        else if (type == 1) rc = inf_fixed(s, lc, dc, lens);
        else if (type == 2) rc = inf_dynamic(s, lc, dc, lens);
        else rc = INF_E_BTYPE;
        if (rc) return rc;
    } while (!last);
    if (s.pos - (uint32_t)(s.cnt >> 3) != n) return INF_E_TRAIL;   // whole bytes still buffered were never consumed
    if (s.op != isize) return INF_E_SIZE;
    if (inf_crc32(crc_t, out, isize) != crc) return INF_E_CRC;
    return INF_OK;
}
// INFLATE-HOST-END

namespace {

constexpr int INF_TPB = 64;

// members: [n][5] int64 = payload offset, payload length, ISIZE, CRC-32, output offset (validated by the host)
__global__ void __launch_bounds__(INF_TPB) wfl_inflate_members(const uint8_t *comp, const long long *members, long long n,
                                                              uint8_t *text, int *first_bad) {
    __shared__ uint32_t crc_t[1024];
    if (threadIdx.x == 0) inf_crc_tables(crc_t);
    __syncthreads();
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    InfHuff lc, dc;
    uint8_t lens[320];
    const long long *r = members + 5 * m;
    const int rc = inf_member(comp + r[0], (uint32_t)r[1], text + r[4], (uint32_t)r[2], (uint32_t)r[3], crc_t, lc, dc, lens);
    if (rc != INF_OK) atomicMin(first_bad, (int)m);
}

}  // namespace
}  // namespace wfl

using namespace wfl;

extern "C" {

/* Inflate a BGZF file's members into the parser's resident text (see the header).  Returns the text length, or a
 * negative wfl_status: WFL_ERR_DATA when a member fails validation (*bad_member = the first such member). */
int64_t wfl_inflate_bgzf(wfl_parser *p, const uint8_t *comp, int64_t comp_len, const int64_t *members, int64_t n_members,
                         int64_t *bad_member, float *ms_h2d, float *ms_kernel) {
    if (!p || (!comp && comp_len) || comp_len < 0 || n_members < 0 || (!members && n_members) || n_members > 2147483647ll)
        return WFL_ERR_ARG;
    if (bad_member) *bad_member = -1;
    // the member table comes from the caller: every payload inside `comp`, members <= 64 KB, outputs tiling the text
    long long total = 0;
    for (long long m = 0; m < n_members; ++m) {
        const int64_t *r = members + 5 * m;
        if (r[0] < 0 || r[1] < 0 || r[1] > 0xffffffffll || r[0] > comp_len - r[1] || r[2] < 0 || r[2] > 65536 ||
            r[3] < 0 || r[3] > 0xffffffffll || r[4] != total) {
            snprintf(p->err, sizeof p->err, "wfl_inflate_bgzf: member %lld of the table is inconsistent", m);
            return WFL_ERR_ARG;
        }
        total += r[2];
    }
    PCU(cudaSetDevice(p->device));
    p->n_rows = 0;
    p->blast_ok = p->genes_ok = false;
    p->text_bytes = 0;
    int rc;
    if ((rc = pensure(p, p->text, (size_t)total + 64)) || (rc = pensure(p, p->comp, (size_t)comp_len)) ||
        (rc = pensure(p, p->mtab, (size_t)n_members * 40)) || (rc = pensure(p, p->counters, 16)))
        return rc;
    PCU(cudaEventRecord(p->ev[0], p->stream));
    if (comp_len) PCU(cudaMemcpyAsync(p->comp.p, comp, (size_t)comp_len, cudaMemcpyHostToDevice, p->stream));
    if (n_members) PCU(cudaMemcpyAsync(p->mtab.p, members, (size_t)n_members * 40, cudaMemcpyHostToDevice, p->stream));
    const int init = 2147483647;
    PCU(cudaMemcpyAsync(p->counters.p, &init, 4, cudaMemcpyHostToDevice, p->stream));
    PCU(cudaEventRecord(p->ev[1], p->stream));
    if (n_members)
        wfl_inflate_members<<<(unsigned)((n_members + INF_TPB - 1) / INF_TPB), INF_TPB, 0, p->stream>>>(
            static_cast<const uint8_t *>(p->comp.p), static_cast<const long long *>(p->mtab.p), n_members,
            static_cast<uint8_t *>(p->text.p), static_cast<int *>(p->counters.p));
    PCU(cudaGetLastError());
    PCU(cudaEventRecord(p->ev[2], p->stream));
    int first_bad = 0;
    PCU(cudaMemcpyAsync(&first_bad, p->counters.p, 4, cudaMemcpyDeviceToHost, p->stream));
    PCU(cudaStreamSynchronize(p->stream));
    float h2d = 0, kern = 0;
    PCU(cudaEventElapsedTime(&h2d, p->ev[0], p->ev[1]));
    PCU(cudaEventElapsedTime(&kern, p->ev[1], p->ev[2]));
    if (ms_h2d) *ms_h2d = h2d;
    if (ms_kernel) *ms_kernel = kern;
    if (first_bad != 2147483647) {
        if (bad_member) *bad_member = first_bad;
        snprintf(p->err, sizeof p->err, "BGZF member %d failed validation on the device", first_bad);
        return WFL_ERR_DATA;
    }
    p->text_bytes = total;
    return total;
}

}  // extern "C"
