"""CPU: compressed blastouts.  BGZF classification and member tables (waafle_b200/compressed.py), chunk ownership over
BGZF text, the streaming reader of generic gzip / bzip2, the BGZF member decoder of csrc/wfl_inflate.cu built for the
host with the address and undefined-behaviour sanitizers against zlib, and streamed runs (two workers, the numpy-oracle
engine, --cpu-parse) on text, BGZF, gzip and bzip2 blastouts giving the same bytes."""
import bz2
import functools
import gzip
import os
import random
import struct
import subprocess
import zlib

import numpy as np
import pytest

import helpers
from test_streaming import OracleEngine, same_outputs, single_pass
from waafle_b200 import compressed, orgscorer, parsers, streaming, synth, taxonomy
from waafle_b200.utils import read_contig_lengths

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(os.path.dirname(HERE), "waafle_b200", "csrc", "wfl_inflate.cu")
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


# ---- a BGZF writer (Python has no bgzip) ----------------------------------------------------------------------------

def raw_deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush_every=0):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    if not flush_every:
        return c.compress(data) + c.flush()
    out = b""
    for k in range(0, len(data), flush_every):   # a full flush ends a block: several blocks per member
        out += c.compress(data[k:k + flush_every]) + c.flush(zlib.Z_FULL_FLUSH)
    return out + c.flush()


def bgzf_member(data, **kw):
    payload = raw_deflate(data, **kw)
    head = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, len(payload) + 25)
    return head + payload + struct.pack("<II", zlib.crc32(data), len(data))


def bgzf(data, block=65280, eof=True, cuts=None, **kw):
    """BGZF bytes of `data`: members of `block` bytes, or split at the offsets `cuts` (and within pieces over `block`)."""
    edges = [0] + (list(cuts) if cuts is not None else []) + [len(data)]
    pieces = [(k, min(k + block, b)) for a, b in zip(edges[:-1], edges[1:]) for k in range(a, max(b, a + 1), block)]
    out = b"".join(bgzf_member(data[a:b], **kw) for a, b in pieces)
    return out + (BGZF_EOF if eof else b"")


# ---- classification and member tables ---------------------------------------------------------------------------

def test_member_table_of_bgzf(tmp_path):
    data = bytes(random.Random(1).getrandbits(8) for _ in range(200000))
    raw = bgzf(data, block=50000)
    members = compressed.bgzf_members(raw)
    assert members.shape == (5, 5)   # 4 data members + the EOF member
    assert list(members[:, compressed.ISIZE]) == [50000] * 4 + [0]
    assert list(members[:, compressed.OUT_OFF]) == [0, 50000, 100000, 150000, 200000]
    for m in range(4):
        o, n = members[m, compressed.PAYLOAD_OFF], members[m, compressed.PAYLOAD_LEN]
        piece = zlib.decompress(raw[o:o + n], wbits=-15)
        assert piece == data[50000 * m:50000 * (m + 1)] and zlib.crc32(piece) == members[m, compressed.CRC]
    assert compressed.member_starts(members)[1] == members[0, compressed.PAYLOAD_OFF] + members[0, compressed.PAYLOAD_LEN] + 8
    path = tmp_path / "x.blastout.gz"
    path.write_bytes(raw)
    kind, table = compressed.classify(str(path))
    assert kind == compressed.BGZF and np.array_equal(table, members)
    assert gzip.decompress(raw) == data   # what the host path reads


def test_generic_gzip_and_suffixes(tmp_path):
    data = b"a\tb\n" * 5000
    single = gzip.compress(data)
    cases = {"one.gz": single, "cat.gz": single + gzip.compress(data),   # `gzip`, `cat a.gz b.gz`
             "trunc.gz": bgzf(data, block=4000)[:-40],                     # BSIZE chain runs past the end
             "short.gz": bgzf(data, block=4000) + b"\x1f\x8b",              # bytes after the chain
             "empty.gz": b""}
    for name, raw in cases.items():
        (tmp_path / name).write_bytes(raw)
        assert compressed.classify(str(tmp_path / name)) == (compressed.GZIP, None), name
    # bgzip's EOF member alone, and a file of one member without it
    assert compressed.bgzf_members(BGZF_EOF).tolist() == [[18, 2, 0, 0, 0]]
    assert compressed.bgzf_members(bgzf(data, block=1 << 16, eof=False)).shape == (1, 5)
    # headers that do not follow the format: another FLG, a missing BC subfield, a second BC, an ISIZE over 64 KB
    good = bgzf_member(data[:1000])
    assert compressed.bgzf_members(good[:3] + b"\x0c" + good[4:]) is None
    assert compressed.bgzf_members(good[:12] + b"XC" + good[14:]) is None
    two_bc = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", 12) + (b"BC" + struct.pack("<HH", 2, len(good) + 5)) * 2
    assert compressed.bgzf_members(two_bc + good[18:]) is None
    assert compressed.bgzf_members(good[:-4] + struct.pack("<I", 70000)) is None
    (tmp_path / "x.bz2").write_bytes(bz2.compress(data))
    (tmp_path / "x.blastout").write_bytes(data)
    assert compressed.classify(str(tmp_path / "x.bz2")) == (compressed.BZIP2, None)
    assert compressed.classify(str(tmp_path / "x.blastout")) == (compressed.TEXT, None)


# ---- chunk ownership over BGZF text -----------------------------------------------------------------------------

def _blast_text(n_contigs=60, seed=3):
    data = synth.generate_config("cfg2", n_contigs=n_contigs, seed=seed)
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        return open(data.write_files(d, "s")["blastout"], "rb").read()


def _assert_tiles_by_blocks(text, chunks):
    assert chunks[0][0] == 0 and sum(n for _, n in chunks) == len(text)
    pos, seen = 0, set()
    for off, n in chunks:
        assert off == pos and n > 0
        pos += n
        assert off == 0 or text[off - 1:off] == b"\n"
        names = {r.split(b"\t")[0] for r in text[off:off + n].split(b"\n") if r}
        assert not names & seen   # a contig block is never split
        seen |= names


def test_bgzf_chunks_tile_the_text_and_never_split_a_block():
    text = _blast_text()
    rows = text.split(b"\n")
    starts = np.cumsum([0] + [len(r) + 1 for r in rows[:-1]])
    changes = [int(s) for k, s in enumerate(starts[1:], 1) if rows[k] and rows[k].split(b"\t")[0] != rows[k - 1].split(b"\t")[0]]
    layouts = {
        "mid-row": [int(s) + 7 for s in starts[5:-1:9]],
        "row start": [int(s) for s in starts[3:-1:11]],
        "query change": changes[::2],
        "tiny members": list(range(37, len(text), 37)),     # members much smaller than rows
        "large": list(range(65000, len(text), 65000)),
    }
    for name, cuts in layouts.items():
        raw = bgzf(text, cuts=sorted(set(c for c in cuts if 0 < c < len(text))))
        members = compressed.bgzf_members(raw)
        reader = compressed.BgzfReader(raw, members)
        assert reader.size == len(text)
        for target in (1, 500, 4096, 30000, len(text) + 1):   # chunks of one block each, blocks longer than a chunk, one chunk
            chunks = streaming.scan_text_chunks(reader, reader.size, target)
            assert chunks == streaming.scan_text_chunks(_FileLike(text), len(text), target), (name, target)
            _assert_tiles_by_blocks(text, chunks)
            for off, n in chunks:   # the members a worker inflates hold its bytes
                m0, m1 = compressed.member_range(members, off, n)
                comp, sub = compressed.sub_table(raw, members, m0, m1)
                own = off - int(members[m0, compressed.OUT_OFF])
                assert gzip.decompress(comp)[own:own + n] == text[off:off + n]
                assert sub[0, compressed.OUT_OFF] == 0 and own + n <= compressed.text_size(sub)


class _FileLike:
    def __init__(self, data):
        self.data, self.pos = data, 0

    def seek(self, pos):
        self.pos = pos

    def read(self, n):
        out = self.data[self.pos:self.pos + n]
        self.pos += len(out)
        return out


# ---- the streaming reader of generic gzip / bzip2 -----------------------------------------------------------------

@pytest.mark.parametrize("suffix", [".gz", ".bz2"])
def test_stream_text_chunks_cut_at_query_changes(tmp_path, suffix):
    text = _blast_text(n_contigs=80, seed=9)
    path = tmp_path / ("x.blastout" + suffix)
    path.write_bytes(gzip.compress(text) if suffix == ".gz" else bz2.compress(text))
    for target in (1, 3000, 50000, len(text) * 2):
        pieces = list(streaming.stream_text_chunks(str(path), target))
        assert b"".join(pieces) == text
        off, chunks = 0, []
        for p in pieces:
            chunks.append((off, len(p)))
            off += len(p)
        _assert_tiles_by_blocks(text, chunks)
        if target == 1:   # every query change is a cut
            assert len(pieces) == len({r.split(b"\t")[0] for r in text.split(b"\n") if r})


# ---- the decoder, built for the host, against zlib ---------------------------------------------------------------

def _zlib_verdict(payload, isize, crc):
    """The member's text if zlib accepts it exactly as a BGZF member (stream ends at the payload's end, ISIZE, CRC)."""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(payload)
    except zlib.error:
        return None
    if not d.eof or d.unused_data or len(out) != isize or zlib.crc32(out) != crc:
        return None
    return out


def _payloads(rng):
    text = open(os.path.join(helpers.GOLDEN, "demo", "demo_contigs.blastout"), "rb").read()
    rand = bytes(rng.getrandbits(8) for _ in range(65536))
    block = rand[:32768]
    yield text[:65280]
    yield text[100000:100000 + 4000]
    yield rand                                            # incompressible: stored blocks at level 0, Huffman-only otherwise
    yield b"a" * 65536                                    # distance-1 overlaps, length-258 matches
    yield block + block                                   # distance 32768
    yield (b"ACGT" * 300 + rand[:50]) * 40                # short periods, overlapping matches
    yield b""                                             # an empty member
    yield b"x"
    yield bytes(rng.choice(b"ACGT\t\n|=.0123456789") for _ in range(60000))


def _corpus(rng):
    """(payload, isize, crc, expected text or None): zlib output at every level and strategy, multi-block members, then
    corruptions of them -- bit flips (anywhere, and in a dynamic block's code-length header), truncations, bytes appended,
    distances before the member's start, ISIZE and CRC mismatches."""
    good = []
    for data in _payloads(rng):
        for level in (0, 1, 6, 9):
            good.append((raw_deflate(data, level), data))
        for strategy in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED):
            good.append((raw_deflate(data, 6, strategy), data))
        if len(data) > 20000:
            good.append((raw_deflate(data, 6, flush_every=7000), data))
            good.append((raw_deflate(data, 0, flush_every=9000), data))
    cases = [(p, len(d), zlib.crc32(d), d) for p, d in good]
    for p, d in good:
        crc = zlib.crc32(d)
        cases.append((p, len(d) + 1, crc, None))
        if d:
            cases.append((p, len(d) - 1, crc, None))
        cases.append((p, len(d), crc ^ 1, None))
        cases.append((p + b"\0", len(d), crc, None))
        for cut in {0, 1, len(p) // 2, max(len(p) - 1, 0)}:
            cases.append((p[:cut], len(d), crc, None))
        for _ in range(40):
            q = bytearray(p)
            if not q:
                break
            span = min(len(q), 24) if rng.random() < 0.5 else len(q)   # half of them in the block header
            q[rng.randrange(span)] ^= 1 << rng.randrange(8)
            cases.append((bytes(q), len(d), crc, None))
    # distances before the start: a stream compressed against a preset dictionary
    text = open(os.path.join(helpers.GOLDEN, "demo", "demo_contigs.blastout"), "rb").read()
    for k in range(8):
        piece = text[20000 * k:20000 * k + 3000]
        c = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY, zdict=text[20000 * k - 30000:20000 * k] or text[-30000:])
        cases.append((c.compress(piece) + c.flush(), len(piece), zlib.crc32(piece), None))
    # hand-made headers: block type 3, a stored block with LEN != ~NLEN, a dynamic header whose code-length code is
    # over-subscribed, and literal/length 286 and distance 30 in fixed blocks
    cases.append((b"\x07\x00", 0, 0, None))
    cases.append((b"\x01\x05\x00\xfb\xfe" + b"abcde", 5, zlib.crc32(b"abcde"), None))
    cases.append((bytes([0x05, 0xe0, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff]), 0, 0, None))
    return [(p, isize, crc, _zlib_verdict(p, isize, crc) if want is None else want) for p, isize, crc, want in cases]


def test_decoder_on_host_against_zlib(tmp_path):
    src = open(SRC).read()
    region = src[src.index("// INFLATE-HOST-BEGIN"):src.index("// INFLATE-HOST-END")]
    (tmp_path / "inflate_region.inc").write_text(region)
    exe = str(tmp_path / "inflate_host")
    cc = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.run([cc, "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-I", str(tmp_path), os.path.join(HERE, "host_inflate", "inflate_host.cpp"), "-o", exe], check=True)
    rng = random.Random(2024)
    cases = _corpus(rng)
    n_reject = sum(want is None for *_, want in cases)
    assert len(cases) > 4000 and n_reject > 3000
    blob = [struct.pack("<I", len(cases))]
    for payload, isize, crc, want in cases:
        blob.append(struct.pack("<I", len(payload)) + payload + struct.pack("<IIB", isize, crc, want is not None))
        if want is not None:
            blob.append(want)
    (tmp_path / "corpus.bin").write_bytes(b"".join(blob))
    out = subprocess.run([exe, str(tmp_path / "corpus.bin")], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert " 0 mismatches" in out.stdout


# ---- streamed runs on compressed blastouts (two workers, the numpy oracle as the engine, --cpu-parse) ----------------

def _compress_variants(path, outdir):
    """The blastout as text, BGZF, one gzip member and bzip2, written under `outdir`."""
    text = open(path, "rb").read()
    out = {"text": path}
    for kind, name, raw in (("bgzf", "x.blastout.gz", bgzf(text, block=3000)), ("gzip", "y.blastout.gz", gzip.compress(text)),
                            ("bz2", "x.blastout.bz2", bz2.compress(text))):
        out[kind] = os.path.join(str(outdir), name)
        with open(out[kind], "wb") as fh:
            fh.write(raw)
    assert compressed.classify(out["bgzf"])[0] == compressed.BGZF
    assert compressed.classify(out["gzip"])[0] == compressed.GZIP
    return out


def _streamed_cli(files, blastout, outdir, flags, chunk_bytes):
    argv = [files["contigs"], blastout, files["gff"], files["taxonomy"], "--outdir", str(outdir), "--basename", "run",
            "--cpu-parse", "--quiet"] + flags
    args = orgscorer.get_args(argv)
    tax = taxonomy.Taxonomy(files["taxonomy"])
    lengths = read_contig_lengths(files["contigs"])
    loci = parsers.read_gff_loci(files["gff"])
    stats, n_chunks = streaming.run_streaming(args, tax, lengths, loci, functools.partial(orgscorer.params_from_args, args),
                                              [0, 0], chunk_bytes, engine_factory=OracleEngine)
    assert not [f for f in os.listdir(str(outdir)) if f.startswith("wfl_shards_")]
    return n_chunks


@pytest.mark.parametrize("shape", ["demo", "cfg5"])
def test_streamed_compressed_blastouts_give_the_same_bytes(tmp_path, shape):
    if shape == "demo":
        files = helpers.demo_files(tmp_path, False)
        flags, cli = {}, []
    else:
        data = synth.generate_config("cfg5", n_contigs=90, seed=77, annotations=True)
        files = data.write_files(str(tmp_path), "s")
        flags, cli = dict(weak_loci="assign-unknown"), ["--weak-loci", "assign-unknown"]
    ref = tmp_path / "single"
    ref.mkdir()
    single_pass(files, str(ref), flags)
    chunk = max(1, os.path.getsize(files["blastout"]) // 6)
    for kind, path in _compress_variants(files["blastout"], tmp_path).items():
        out = tmp_path / kind
        out.mkdir()
        n = _streamed_cli(files, path, out, cli, chunk)
        assert n >= 4, kind
        same_outputs(str(ref), str(out))


def test_streamed_corrupt_gzip_raises_the_gzip_error(tmp_path):
    files = helpers.demo_files(tmp_path, False)
    text = open(files["blastout"], "rb").read()
    raw = bytearray(gzip.compress(text))
    raw[-6] ^= 0xff   # the trailer's CRC
    bad = tmp_path / "bad.blastout.gz"
    bad.write_bytes(bytes(raw))
    out = tmp_path / "out"
    out.mkdir()
    with pytest.raises(gzip.BadGzipFile):
        _streamed_cli(files, str(bad), out, [], 4000)
    assert not [f for f in os.listdir(str(out)) if f.startswith("wfl_shards_")]
