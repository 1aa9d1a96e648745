"""GPU: BGZF blastouts inflated on the device (csrc/wfl_inflate.cu).  The device's text equals zlib's byte for byte;
members that fail validation come back as the first failing member and send the CLI to the host reader, which raises
gzip's error; `parse_bgzf` equals `parse` on the same text; and the CLIs write the same bytes from a BGZF blastout as
from the plain text -- single call, streamed on one device and on `--devices 0,0` -- while reporting that the device
inflated it (so a BGZF fixture cannot pass on the host path)."""
import gzip
import json
import os
import random
import zlib

import numpy as np
import pytest

import helpers
from test_compressed import BGZF_EOF, _payloads, bgzf, bgzf_member, raw_deflate
from waafle_b200 import compressed, gpu_parse, synth

pytestmark = pytest.mark.gpu
DEVICE_ROUTE, STREAM_ROUTE = "members inflated on cuda:", "BGZF members inflated on the device"


@pytest.fixture(scope="module")
def parser():
    p = gpu_parse.BlastParser(0)
    yield p
    p.close()


def _good_members(rng):
    out = []
    for data in _payloads(rng):
        data = data[:65280]   # a BGZF member holds at most 64 KB, compressed too
        for level in (0, 1, 6, 9):
            out.append(bgzf_member(data, level=level))
        for strategy in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED):
            out.append(bgzf_member(data, strategy=strategy))
        if len(data) > 20000:
            out.append(bgzf_member(data, flush_every=7000))
    return out


def test_device_inflate_equals_zlib(parser):
    raw = b"".join(_good_members(random.Random(7))) + BGZF_EOF
    members = compressed.bgzf_members(raw)
    n = parser.inflate_bgzf(raw, members)
    want = gzip.decompress(raw)
    assert n == len(want) and bytes(parser.text(0, n)) == want
    assert bytes(parser.text(1000, 77)) == want[1000:1077]
    # a cfg2-shape blastout at level 6
    data = synth.generate_config("cfg2", n_contigs=3000, seed=11)
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        text = open(data.write_files(d, "s")["blastout"], "rb").read()
    raw = bgzf(text)
    members = compressed.bgzf_members(raw)
    assert len(members) > 100
    n = parser.inflate_bgzf(raw, members)
    assert n == len(text) and bytes(parser.text(0, n)) == text


def _corrupt_cases():
    """(name, BGZF bytes, index of the bad member): one bad member among good ones."""
    text = open(os.path.join(helpers.GOLDEN, "demo", "demo_contigs.blastout"), "rb").read()
    step = len(text) // 10
    pieces = [text[k * step:(k + 1) * step] for k in range(10)]
    good = [bgzf_member(p) for p in pieces]
    cases = []

    def with_member(k, member):
        return (b"".join(good[:k] + [member] + good[k + 1:]) + BGZF_EOF, k)

    m = bytearray(good[3])
    m[-8] ^= 1   # trailer CRC
    cases.append(("crc",) + with_member(3, bytes(m)))
    m = bytearray(good[6])
    m[40] ^= 0x10   # a bit of the payload
    cases.append(("bit flip",) + with_member(6, bytes(m)))
    c = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY, zdict=pieces[0])
    payload = c.compress(pieces[1]) + c.flush()   # matches reach into the previous member
    head = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\x00BC\x02\x00" + (len(payload) + 25).to_bytes(2, "little")
    cases.append(("distance before start",) + with_member(
        2, head + payload + zlib.crc32(pieces[1]).to_bytes(4, "little") + len(pieces[1]).to_bytes(4, "little")))
    m = bytearray(good[8])
    m[-4:] = (len(pieces[8]) - 1).to_bytes(4, "little")   # ISIZE one short
    cases.append(("isize",) + with_member(8, bytes(m)))
    payload = raw_deflate(pieces[4])[:-3]   # the stream stops short of its end
    head = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\x00BC\x02\x00" + (len(payload) + 25).to_bytes(2, "little")
    cases.append(("truncated",) + with_member(
        4, head + payload + zlib.crc32(pieces[4]).to_bytes(4, "little") + len(pieces[4]).to_bytes(4, "little")))
    m = bytearray(good[1])
    m[18] = (m[18] & 1) | 0x06   # block type 3
    cases.append(("block type",) + with_member(1, bytes(m)))
    return cases


def test_corrupt_members_are_reported(parser, tmp_path):
    for name, raw, bad in _corrupt_cases():
        members = compressed.bgzf_members(raw)
        assert members is not None, name
        with pytest.raises(gpu_parse.InflateError) as exc:
            parser.inflate_bgzf(raw, members)
        assert exc.value.member == bad, name
        with pytest.raises(Exception):
            gzip.decompress(raw)   # the host path rejects the same file
    # the parser is usable after a failed inflate
    raw = bgzf(b"x\ty\n" * 1000)
    assert parser.inflate_bgzf(raw, compressed.bgzf_members(raw)) == 4000


def test_corrupt_bgzf_cli_takes_the_host_path(tmp_path, capfd):
    """A member that fails on the device sends the file to the host reader: the run ends exactly as with --cpu-parse
    (gzip's error, or the outputs when the host reader does not check what the device rejected)."""
    from waafle_b200 import orgscorer
    files = helpers.demo_files(tmp_path, False)
    for name, raw, bad in _corrupt_cases()[:3]:
        path = str(tmp_path / "bad.blastout.gz")
        with open(path, "wb") as fh:
            fh.write(raw)
        outcome = {}
        for tag, extra in (("gpu", []), ("host", ["--cpu-parse"])):
            out = tmp_path / (tag + name.replace(" ", "_"))
            out.mkdir()
            try:
                orgscorer.main([files["contigs"], path, files["gff"], files["taxonomy"], "--outdir", str(out),
                                "--basename", "run", "--quiet"] + extra)
                outcome[tag] = _outputs(out)
            except BaseException as exc:   # noqa: B902 -- SystemExit and gzip's errors alike
                outcome[tag] = (type(exc), str(exc))
            if tag == "gpu":
                assert "BGZF member {} failed validation".format(bad) in capfd.readouterr().err, name
        assert outcome["gpu"] == outcome["host"], name


def _blast_text(n_contigs, seed, shape="cfg2"):
    import tempfile
    data = synth.generate_config(shape, n_contigs=n_contigs, seed=seed, annotations=True)
    with tempfile.TemporaryDirectory() as d:
        return open(data.write_files(d, "s")["blastout"], "rb").read()


def _same_tables(a, b):
    for f in ("qstart", "qend", "score", "scov_modified", "strand", "sysmask", "block_starts"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert np.array_equal(a.taxon, b.taxon)   # codes are hash-slot ranks: the names they stand for are the contract
    assert sorted(a.taxon_names) == sorted(b.taxon_names) and a.systems == b.systems and list(a.block_names) == list(b.block_names)
    assert [a.sseqid_names[i] for i in range(0, len(a), 97)] == [b.sseqid_names[i] for i in range(0, len(b), 97)]


def test_parse_bgzf_equals_parse(parser):
    text = _blast_text(600, 12)
    raw = bgzf(text, block=20000)
    members = compressed.bgzf_members(raw)
    want = parser.parse(text)
    genes_want = parser.call_genes(0.1, 90, 0.75)
    got = parser.parse_bgzf(raw, members)
    genes_got = parser.call_genes(0.1, 90, 0.75)
    _same_tables(got, want)
    for x, y in zip(genes_got, genes_want):
        assert np.array_equal(x, y)
    # an owned range (whole rows, not starting at a member boundary)
    rows = text.split(b"\n")
    off = sum(len(r) + 1 for r in rows[:1234])
    n = sum(len(r) + 1 for r in rows[1234:4321])
    _same_tables(parser.parse_bgzf(raw, members, own=(off, n)), parser.parse(text[off:off + n]))
    assert len(parser.parse_bgzf(raw, members, own=(off, 0))) == 0


# ---- the CLIs on a BGZF blastout ------------------------------------------------------------------------------------

ROUTES = (("single", []), ("stream", ["--stream-mb", "0.02"]), ("devices", ["--stream-mb", "0.02", "--devices", "0,0"]))


def _outputs(outdir, details=False):
    got = {k: open(os.path.join(str(outdir), "run.{}.tsv".format(k))).read() for k in ("lgt", "no_lgt", "unclassified")}
    if details:
        with gzip.open(os.path.join(str(outdir), "run.details.tsv.gz"), "rt") as fh:
            got["details"] = fh.read()
    return got


def _check_route(capfd, route):
    err = capfd.readouterr().err
    assert (DEVICE_ROUTE if route == "single" else STREAM_ROUTE) in err, err[-2000:]


def _bgzf_copy(path, outdir, block=7000):
    out = os.path.join(str(outdir), "bgzf.blastout.gz")
    with open(path, "rb") as fh, open(out, "wb") as dst:
        dst.write(bgzf(fh.read(), block=block))
    assert compressed.classify(out)[0] == compressed.BGZF
    return out


def _shapes(tmp_path):
    os.makedirs(str(tmp_path / "demo"))
    demo = helpers.demo_files(tmp_path / "demo", False)
    data = synth.generate_config("cfg5", n_contigs=300, seed=402, annotations=True)
    os.makedirs(str(tmp_path / "cfg5"))
    cfg5 = data.write_files(str(tmp_path / "cfg5"), "run")
    flag_sets = json.load(open(os.path.join(helpers.GOLDEN, "demo_cli", "flag_sets.json")))
    return [("demo", demo, flag_sets), ("cfg5", cfg5, [["--weak-loci", "assign-unknown"]])]


def test_orgscorer_bgzf_equals_text(tmp_path, capfd):
    from waafle_b200 import orgscorer
    for shape, files, flag_sets in _shapes(tmp_path):
        gz = _bgzf_copy(files["blastout"], os.path.dirname(files["contigs"]))
        for k, flags in enumerate(flag_sets):
            for mode, extra in (("fast", []), ("exact", ["--exact-scores"]), ("details", ["--write-details"])):
                if k and mode != "fast":
                    continue
                for route, rflags in ROUTES:
                    outs = {}
                    for tag, blastout in (("text", files["blastout"]), ("bgzf", gz)):
                        out = tmp_path / "o_{}_{}_{}_{}_{}".format(shape, k, mode, route, tag)
                        out.mkdir()
                        orgscorer.main([files["contigs"], blastout, files["gff"], files["taxonomy"], "--outdir", str(out),
                                        "--basename", "run"] + flags + extra + rflags)
                        if tag == "bgzf":
                            _check_route(capfd, route)
                        outs[tag] = _outputs(out, details=mode == "details")
                    assert outs["text"] == outs["bgzf"], (shape, flags, mode, route)


def test_pipeline_and_genecaller_bgzf_equal_text(tmp_path, capfd):
    from waafle_b200 import genecaller, pipeline
    for shape, files, flag_sets in _shapes(tmp_path):
        gz = _bgzf_copy(files["blastout"], os.path.dirname(files["contigs"]))
        for route, rflags in ROUTES:
            outs = {}
            for tag, blastout in (("text", files["blastout"]), ("bgzf", gz)):
                out = tmp_path / "p_{}_{}_{}".format(shape, route, tag)
                out.mkdir()
                gff = str(out / "calls.gff")
                pipeline.main([files["contigs"], blastout, files["taxonomy"], "--outdir", str(out), "--basename", "run",
                               "--gff", gff] + flag_sets[0] + rflags)
                if tag == "bgzf":
                    _check_route(capfd, route)
                outs[tag] = _outputs(out)
                outs[tag]["gff"] = open(gff).read()
            assert outs["text"] == outs["bgzf"], (shape, route)
        gffs = []
        for tag, blastout in (("text", files["blastout"]), ("bgzf", gz)):
            gff = str(tmp_path / "g_{}_{}.gff".format(shape, tag))
            genecaller.main([blastout, "--gff", gff])
            gffs.append(open(gff).read())
            if tag == "bgzf":
                _check_route(capfd, "single")
        assert gffs[0] == gffs[1] and gffs[0].count("\n") > 10, shape
