"""BGZF blastouts inflated on the device: kernel rate, copies and what the pipeline CLI gains, on a cfg2-shape workload.

    python tools/inflate_timing.py [--contigs 100000] [--repeats 3] [--devices all] [--out profiles/inflate_cfg2.json]

The cfg2 shape (--contigs contigs) is written as text files, and its blastout also as BGZF (64 KB members, zlib level 6,
what bgzip writes) and as one gzip member (level 6, what `gzip` writes).
1. In process: wfl_inflate_bgzf over the whole file (CUDA events; the median of 5 after a warm-up): H2D bytes and time,
   kernel time, GB/s of text; the device text is compared with zlib's.  For scale, one host core's gzip.decompress.
2. The blastout read of the fused pipeline (parsers.read_blast_hits_and_genes) for text, BGZF and gzip: wall time and
   the parser's stage times.
3. `python -m waafle_b200.pipeline` wall time for text, BGZF and gzip, alternating, median of --repeats; the outputs
   must be byte-identical.  Then the streamed run (--stream-mb 256) on one GPU and on --devices, text and BGZF.

One JSON line goes to --out, with the card name and power limit read in the same run.
"""
import argparse
import concurrent.futures
import gzip
import json
import os
import struct
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    if not out:
        raise SystemExit("no GPU visible: this measurement needs one")
    return [ln.strip() for ln in out]


def bgzf_member(data, level):
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    payload = c.compress(data) + c.flush()
    head = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, len(payload) + 25)
    return head + payload + struct.pack("<II", zlib.crc32(data), len(data))


def write_bgzf(text, path, level=6, block=65280):
    with concurrent.futures.ThreadPoolExecutor(os.cpu_count()) as ex, open(path, "wb") as fh:
        for m in ex.map(lambda k: bgzf_member(text[k:k + block], level), range(0, len(text), block), chunksize=64):
            fh.write(m)
        fh.write(BGZF_EOF)


def progress(*args):
    print(*args, file=sys.stderr, flush=True)


def median(x):
    x = sorted(x)
    return x[len(x) // 2]


def device_inflate(path, text):
    from waafle_b200 import compressed, gpu_parse
    comp = open(path, "rb").read()
    kind, members = compressed.classify(path)
    assert kind == compressed.BGZF
    p = gpu_parse.BlastParser(0)
    runs = []
    for r in range(6):
        n = p.inflate_bgzf(comp, members)
        if r:
            runs.append(dict(p.inflate_times))
    same = bytes(p.text(0, n)) == text
    p.close()
    ms_k = median([t["ms_inflate"] for t in runs])
    ms_h = median([t["ms_h2d"] for t in runs])
    t = time.perf_counter()
    host = gzip.decompress(comp)
    s_host = time.perf_counter() - t
    assert host == text
    return dict(members=len(members), comp_bytes=len(comp), text_bytes=n, ratio=round(n / len(comp), 2),
                ms_kernel=round(ms_k, 2), text_gb_per_s=round(n / ms_k / 1e6, 2), ms_h2d=round(ms_h, 2),
                h2d_gb_per_s=round(len(comp) / ms_h / 1e6, 2), kernel_runs_ms=[round(t["ms_inflate"], 2) for t in runs],
                device_text_equals_zlib=same, s_host_one_core_gzip_decompress=round(s_host, 3))


def read_stage(paths):
    from waafle_b200 import parsers
    out = {}
    for tag, path in paths.items():
        t = time.perf_counter()
        hits, genes = parsers.read_blast_hits_and_genes(path, 0.1, 90, 0.0, device=0)
        s = time.perf_counter() - t
        out[tag] = dict(s_read_parse_genes=round(s, 3), hits=len(hits),
                        parser_ms={k: round(v, 2) for k, v in getattr(hits, "parse_times", {}).items()
                                   if isinstance(v, float)})
    return out


def run_pipeline(files, blastout, outdir, extra):
    os.makedirs(outdir, exist_ok=True)
    cmd = [sys.executable, "-m", "waafle_b200.pipeline", files["contigs"], blastout, files["taxonomy"], "--outdir", outdir,
           "--basename", "run", "--quiet"] + extra
    t = time.perf_counter()
    subprocess.run(cmd, cwd=ROOT, check=True, env=dict(os.environ, PYTHONPATH=ROOT))
    return time.perf_counter() - t


def outputs(outdir):
    return [open(os.path.join(outdir, "run.{}.tsv".format(k)), "rb").read() for k in ("lgt", "no_lgt", "unclassified")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=100000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--devices", default="all")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "inflate_cfg2.json"))
    a = ap.parse_args()
    from waafle_b200 import synth
    result = dict(tool="inflate_timing", workload="cfg2", contigs=a.contigs, gpus=gpu_info())
    with tempfile.TemporaryDirectory() as work:
        t = time.perf_counter()
        files = synth.generate_config("cfg2", n_contigs=a.contigs, seed=1).write_files(os.path.join(work, "in"), "s")
        text = open(files["blastout"], "rb").read()
        paths = dict(text=files["blastout"], bgzf=files["blastout"] + ".bgzf.gz", gzip=files["blastout"] + ".gz")
        progress("cfg2 text written", round(time.perf_counter() - t, 1), "s")
        write_bgzf(text, paths["bgzf"])
        with open(paths["gzip"], "wb") as fh:
            fh.write(gzip.compress(text, 6))
        result["input_generation_s"] = round(time.perf_counter() - t, 1)
        progress("inputs written", result["input_generation_s"], "s")
        result["file_mb"] = {k: round(os.path.getsize(p) / 1e6, 1) for k, p in paths.items()}
        result["device_inflate"] = device_inflate(paths["bgzf"], text)
        del text
        progress("device inflate", result["device_inflate"])
        result["read_stage"] = read_stage(paths)
        progress("read stage", result["read_stage"])
        walls = {k: [] for k in paths}
        for r in range(a.repeats):
            for k, p in paths.items():
                walls[k].append(round(run_pipeline(files, p, os.path.join(work, "cli", k), []), 3))
                progress("pipeline", k, walls[k][-1])
        ref = outputs(os.path.join(work, "cli", "text"))
        result["pipeline_cli"] = dict(median_s={k: median(v) for k, v in walls.items()}, runs_s=walls,
                                      outputs_identical=all(outputs(os.path.join(work, "cli", k)) == ref for k in paths))
        ndev = len(result["gpus"]) if a.devices == "all" else len(a.devices.split(","))
        streamed = {}
        for label, dev in (("1gpu", "0"), ("{}gpu".format(ndev), a.devices)):
            for k in ("text", "bgzf"):
                d = os.path.join(work, "stream", label, k)
                s = run_pipeline(files, paths[k], d, ["--stream-mb", "256", "--devices", dev])
                streamed["{}_{}".format(label, k)] = dict(s=round(s, 3), outputs_identical=outputs(d) == ref)
                progress("streamed", label, k, round(s, 3))
        result["streamed"] = streamed
    line = json.dumps(result)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
