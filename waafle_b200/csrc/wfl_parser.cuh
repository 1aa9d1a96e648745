// The wfl_parser handle, shared by the front-end parsers (wfl_parse.cu) and the gene calls over the blast columns the
// handle keeps on the device (wfl_genecall.cu).
#pragma once

#include <cstdio>
#include <cuda_runtime.h>

#include "waafle_b200.h"

namespace wfl {

// device buffer that only grows (cap = allocated bytes)
struct PBuf {
    void *p = nullptr;
    size_t cap = 0;
};

int pensure(wfl_parser *p, PBuf &b, size_t bytes);   // grows `b` to >= bytes; a wfl_status (text in p->err)

}  // namespace wfl

struct wfl_parser {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {};
    wfl::PBuf gcol[7];
    long long gff_rows = 0;
    wfl::PBuf text, tiles, rows, col[13], tax_hash, tax_off, tax_len, sys_hash, sys_off, sys_len, counters, perm;
    long long n_rows = 0, n_bytes = 0;
    long long text_bytes = 0;         // valid bytes of `text`: the last upload or BGZF inflate
    wfl::PBuf comp, mtab;             // compressed bytes and member table of the last wfl_inflate_bgzf
    bool blast_ok = false;            // col[] holds the last wfl_parse_blast, which flagged no row
    wfl::PBuf gc_pool;                // gene-call scratch and the dense gene arrays of the last wfl_parser_call_genes
    bool genes_ok = false;
    long long gc_blocks = 0, gc_genes = 0;
    float ms_h2d = 0, ms_kernels = 0, ms_d2h = 0;
    char err[256] = {0};
};

#define PCU(call)                                                                                     \
    do {                                                                                              \
        cudaError_t _e = (call);                                                                      \
        if (_e != cudaSuccess) {                                                                      \
            snprintf(p->err, sizeof p->err, "%s failed: %s", #call, cudaGetErrorString(_e));          \
            return WFL_ERR_CUDA;                                                                      \
        }                                                                                             \
    } while (0)
