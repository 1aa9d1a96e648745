// Host build of the BGZF member decoder of waafle_b200/csrc/wfl_inflate.cu (region between the markers
// "INFLATE-HOST-BEGIN" / "INFLATE-HOST-END", extracted by tests/test_compressed.py), built with the address and
// undefined-behaviour sanitizers.  Reads a corpus of members written by the test: every member's payload and output get
// heap buffers of exactly their size, so a read past the payload or a write past ISIZE stops the run.  Each member's
// verdict (accept with the expected bytes, or reject) must equal zlib's.  Exit code 0 = no mismatch.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#define WFL_HD

#include "inflate_region.inc"

static bool rd(FILE *f, void *p, size_t n) { return fread(p, 1, n, f) == n; }

int main(int argc, char **argv) {
    if (argc != 2) return 2;
    FILE *f = fopen(argv[1], "rb");
    if (!f) return 2;
    uint32_t n_cases = 0;
    if (!rd(f, &n_cases, 4)) return 2;
    uint32_t crc_t[1024];
    inf_crc_tables(crc_t);
    InfHuff *lc = new InfHuff, *dc = new InfHuff;
    long bad = 0, accepted = 0, rejected = 0;
    for (uint32_t c = 0; c < n_cases; ++c) {
        uint32_t plen, isize, crc;
        uint8_t ok;
        if (!rd(f, &plen, 4)) return 2;
        uint8_t *payload = static_cast<uint8_t *>(malloc(plen ? plen : 1));
        if (!rd(f, payload, plen) || !rd(f, &isize, 4) || !rd(f, &crc, 4) || !rd(f, &ok, 1)) return 2;
        std::vector<uint8_t> want(ok ? isize : 0);
        if (ok && isize && !rd(f, want.data(), isize)) return 2;
        uint8_t *out = static_cast<uint8_t *>(malloc(isize ? isize : 1));
        uint8_t *lens = static_cast<uint8_t *>(malloc(320));
        const int rc = inf_member(payload, plen, out, isize, crc, crc_t, *lc, *dc, lens);
        const bool same = ok ? rc == INF_OK && (isize == 0 || memcmp(out, want.data(), isize) == 0) : rc != INF_OK;
        if (!same) {
            if (bad < 20) printf("case %u: expected %s, decoder returned %d\n", c, ok ? "accept" : "reject", rc);
            ++bad;
        }
        (rc == INF_OK ? accepted : rejected) += 1;
        free(payload);
        free(out);
        free(lens);
    }
    fclose(f);
    delete lc;
    delete dc;
    printf("%u cases (%ld accepted, %ld rejected), %ld mismatches\n", n_cases, accepted, rejected, bad);
    return bad ? 1 : 0;
}
