"""The pack stage of a GPU-parsed run, host-built batch against device-built batch, on the cfg2 shape written as text.

    python tools/resident_batch_timing.py [--contigs 100000] [--repeats 3] [--outdir profiles]

One parse on the device, then `--repeats` alternations of
  host:     LocusTable.from_blocks, tax.build, packing.pack, orgscorer.score_in_chunks (host columns shipped again)
  resident: LocusTable.from_blocks, tax.build, packing.pack_resident, Engine.score_batch (wfl_upload_parsed)
with the pack wall time, the device time of the batch kernels (ms_kernels of wfl_upload_parsed), the score wall time and
the parser's D2H time of the columns (ms_d2h, paid by both paths).  The three TSVs of the last run of each path must be
equal.  Then the fused CLI (python -m waafle_b200.pipeline) on the same files, median of `--repeats` runs.  Prints one
JSON line and writes it to <outdir>/resident_batch_cfg2.json.  Needs a GPU; its name and power limit are read in the
same run.  The input files go to a temporary directory that is removed at the end."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from waafle_b200 import gpu_parse, orgscorer, packing, parsers, synth, taxonomy, writer   # noqa: E402
from waafle_b200.engine import Engine                                                     # noqa: E402
from waafle_b200.params import OrgscorerParams                                            # noqa: E402
from waafle_b200.utils import read_contig_lengths                                         # noqa: E402

THRESHOLDS = (0.1, 200.0, 0.75)   # genecaller defaults (min_overlap, min_gene_length, min_scov)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def one_path(kind, files, hits, genes, contig_lengths, outdir):
    """One pack + score of the parsed hits; returns the times and writes the TSVs to `outdir`."""
    clock = time.perf_counter
    t0 = clock()
    loci = parsers.LocusTable.from_blocks(list(hits.block_names), *genes)
    tax = taxonomy.Taxonomy(files["taxonomy"])
    tax.build(hits.distinct_taxa())
    batch = (packing.pack_resident if kind == "resident" else packing.pack)(contig_lengths, loci, hits, tax)
    pack_s = clock() - t0
    engine = Engine(0, OrgscorerParams(n_systems=len(hits.systems)), tax)
    t0 = clock()
    res = engine.score_batch(batch) if kind == "resident" else orgscorer.score_in_chunks(engine, batch, 250000)
    score_s = clock() - t0
    ms_kernels = engine.resident_times.get("ms_kernels") if kind == "resident" else None
    engine.close()
    writer.write_main_output_files(writer.build_records(batch, loci, hits, tax, res), outdir, "run")
    return dict(pack_s=round(pack_s, 4), score_s=round(score_s, 4), ms_kernels=ms_kernels)


def outputs(outdir):
    return {k: open(os.path.join(outdir, "run.{}.tsv".format(k)), "rb").read() for k in ("lgt", "no_lgt", "unclassified")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=100000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--outdir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    name, power = gpu_info()
    work = tempfile.mkdtemp(prefix="wfl_resident_timing_")
    try:
        t0 = time.perf_counter()
        data = synth.generate_config("cfg2", n_contigs=args.contigs, seed=2, annotations=False)
        files = data.write_files(work, "run")
        gen_s = time.perf_counter() - t0
        contig_lengths = read_contig_lengths(files["contigs"])
        parser = gpu_parse.BlastParser(0)
        hits = parser.parse(open(files["blastout"], "rb").read())
        assert hits is not None
        ms_d2h = parser.times["ms_d2h"]
        gene_off, start, end, strand = parser.call_genes(*THRESHOLDS)
        genes = (gene_off, start, end, strand)
        runs = {"host": [], "resident": []}
        dirs = {k: os.path.join(work, k) for k in runs}
        for d in dirs.values():
            os.makedirs(d)
        for _ in range(args.repeats):
            for kind in ("host", "resident"):
                assert gpu_parse.live_resident(hits) is not None
                runs[kind].append(one_path(kind, files, hits, genes, contig_lengths, dirs[kind]))
        parser.close()
        equal = outputs(dirs["host"]) == outputs(dirs["resident"])
        fused = []
        for _ in range(args.repeats):
            out = os.path.join(work, "cli")
            os.makedirs(out, exist_ok=True)
            t0 = time.perf_counter()
            subprocess.run([sys.executable, "-m", "waafle_b200.pipeline", files["contigs"], files["blastout"],
                            files["taxonomy"], "--outdir", out, "--basename", "run"], cwd=ROOT, check=True,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            fused.append(round(time.perf_counter() - t0, 3))
        equal_cli = outputs(out) == outputs(dirs["host"])   # the CLI's flags are the defaults used above
        med = lambda kind, key: float(np.median([r[key] for r in runs[kind]]))
        result = dict(
            workload="cfg2", contigs=args.contigs, hits=len(hits), blastout_mb=round(os.path.getsize(files["blastout"]) / 2**20, 1),
            gpu=name, power_limit=power, repeats=args.repeats,
            host_pack_s=med("host", "pack_s"), resident_pack_s=med("resident", "pack_s"),
            host_score_s=med("host", "score_s"), resident_score_s=med("resident", "score_s"),
            resident_ms_kernels=med("resident", "ms_kernels"), parser_ms_d2h=round(ms_d2h, 3),
            runs=runs, outputs_equal=bool(equal), fused_cli_outputs_equal=bool(equal_cli), fused_cli_s=float(np.median(fused)), fused_cli_runs_s=fused,
            input_generation_s=round(gen_s, 1))
    finally:
        shutil.rmtree(work, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    os.makedirs(args.outdir, exist_ok=True)
    with open(os.path.join(args.outdir, "resident_batch_cfg2.json"), "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
