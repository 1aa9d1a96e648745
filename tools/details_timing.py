"""Wall time that --write-details adds to the orgscorer CLI on a cfg2-shape workload, and where it goes.

    python tools/details_timing.py [--contigs 20000] [--big 100000] [--parent-tree DIR] [--out profiles/details_cfg2.json]

1. cfg2 shape, --contigs contigs, written as text files.  The CLI of this tree (and of --parent-tree, a checkout of
   another commit with its library built) runs with and without --write-details, alternating, --repeats times each;
   the added time is the median with-flag run minus the median without-flag run.  The decompressed details tables of
   the two trees must be identical.
2. cfg2 shape, --big contigs, this tree only: rows and text bytes, device time of the text build (CUDA events), D2H,
   compression time and threads, the added wall time, and the same run streamed over --devices (default: every GPU).

One JSON line goes to --out, with the card name and power limit read in the same run.
"""
import argparse
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    if not out:
        raise SystemExit("no GPU visible: this measurement needs one")
    return [ln.strip() for ln in out]


def run_cli(tree, files, outdir, extra):
    os.makedirs(outdir, exist_ok=True)
    cmd = [sys.executable, "-m", "waafle_b200.orgscorer", files["contigs"], files["blastout"], files["gff"],
           files["taxonomy"], "--outdir", outdir, "--basename", "run", "--quiet"] + extra
    t = time.perf_counter()
    subprocess.run(cmd, cwd=tree, check=True, env=dict(os.environ, PYTHONPATH=tree))
    return time.perf_counter() - t


def details(outdir):
    with gzip.open(os.path.join(outdir, "run.details.tsv.gz"), "rb") as fh:
        return fh.read()


def median(x):
    x = sorted(x)
    return x[len(x) // 2]


def added_time(trees, files, work, repeats):
    times = {name: {"with": [], "without": []} for name in trees}
    for r in range(repeats):
        for name, tree in trees.items():
            for flag in ("without", "with"):
                extra = ["--write-details"] if flag == "with" else []
                times[name][flag].append(run_cli(tree, files, os.path.join(work, name, flag), extra))
    out = {}
    for name in trees:
        w, wo = median(times[name]["with"]), median(times[name]["without"])
        out[name] = dict(s_with=round(w, 3), s_without=round(wo, 3), s_added=round(w - wo, 3),
                         runs=times[name])
    return out


def in_process(files, piece_mb):
    """The details run of this tree in one process, timed by stage."""
    from waafle_b200 import packing, parsers, streaming, taxonomy, utils, writer
    from waafle_b200.engine import Engine
    from waafle_b200.params import OrgscorerParams
    from oracle.reference_harness import make_args
    tax = taxonomy.Taxonomy(files["taxonomy"])
    lengths = utils.read_contig_lengths(files["contigs"])
    loci = parsers.read_gff_loci(files["gff"], device=0)
    hits = parsers.read_blast_hits(files["blastout"], device=0)
    tax.build(hits.distinct_taxa())
    batch = packing.pack(lengths, loci, hits, tax)
    params = OrgscorerParams.from_args(make_args(), n_systems=len(hits.systems))
    eng = Engine(0, params, tax)
    eng.score_batch_details(batch, download=False)
    order = streaming.details_order(batch, hits, lengths)
    with tempfile.TemporaryDirectory() as d:
        t = time.perf_counter()
        threads = writer.write_details_file(os.path.join(d, "x.gz"), eng.details_text(order, batch.contig_names,
                                                                                    int(piece_mb * (1 << 20))))
        s_write = time.perf_counter() - t
        gz_bytes = os.path.getsize(os.path.join(d, "x.gz"))
    times = dict(eng.details_times)
    eng.close()
    # compression alone, on the same text (one pass of the thread pool over the whole table)
    eng = Engine(0, params, tax)
    eng.score_batch_details(batch, download=False)
    text = b"".join(eng.details_text(order, batch.contig_names, int(piece_mb * (1 << 20))))
    eng.close()
    with tempfile.TemporaryDirectory() as d:
        t = time.perf_counter()
        writer.write_details_file(os.path.join(d, "y.gz"), [text])
        s_compress = time.perf_counter() - t
    return dict(contigs=batch.n_contigs, hits=batch.n_hits, rows=text.count(b"\n"), text_bytes=len(text),
                gz_bytes=gz_bytes, ms_text_build_device=round(times["ms_length"] + times["ms_text"], 3),
                ms_length_pass=round(times["ms_length"], 3), ms_write_pass=round(times["ms_text"], 3),
                ms_d2h=round(times["ms_d2h"], 3), pieces=times["pieces"], s_text_and_compress=round(s_write, 3),
                s_compress_only=round(s_compress, 3), compress_threads=threads, compress_level=writer.DETAILS_LEVEL)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=20000)
    ap.add_argument("--big", type=int, default=100000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--devices", default="all")
    ap.add_argument("--piece-mb", type=float, default=256.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "details_cfg2.json"))
    a = ap.parse_args()
    from waafle_b200 import synth
    result = dict(tool="details_timing", gpus=gpu_info())
    with tempfile.TemporaryDirectory() as work:
        files = synth.generate_config("cfg2", n_contigs=a.contigs, seed=1).write_files(os.path.join(work, "small"), "s")
        trees = {"this": ROOT}
        if a.parent_tree:
            trees["parent"] = os.path.abspath(a.parent_tree)
        result["small"] = dict(contigs=a.contigs, added=added_time(trees, files, os.path.join(work, "runs"), a.repeats))
        if a.parent_tree:
            same = details(os.path.join(work, "runs", "this", "with")) == details(os.path.join(work, "runs", "parent", "with"))
            p, t = result["small"]["added"]["parent"]["s_added"], result["small"]["added"]["this"]["s_added"]
            result["small"].update(details_identical=same, added_ratio=round(p / t, 1) if t > 0 else None)
        if a.big > 0:
            files = synth.generate_config("cfg2", n_contigs=a.big, seed=1).write_files(os.path.join(work, "big"), "b")
            big = in_process(files, a.piece_mb)
            big["added"] = added_time({"this": ROOT}, files, os.path.join(work, "big_runs"), 1)["this"]
            ndev = len(result["gpus"]) if a.devices == "all" else len(a.devices.split(","))
            s_stream = run_cli(ROOT, files, os.path.join(work, "big_stream"),
                               ["--write-details", "--devices", a.devices, "--stream-mb", "64"])
            one = details(os.path.join(work, "big_runs", "this", "with"))
            big["streamed"] = dict(devices=ndev, s_with_details=round(s_stream, 3),
                                   details_identical=details(os.path.join(work, "big_stream")) == one)
            result["big"] = big
    line = json.dumps(result)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
