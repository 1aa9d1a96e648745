"""CPU: the reference arm of bench.py runs without a GPU and prints its one-line JSON result; --dump-outputs writes the
result arrays within its size limit.  GPU: --steps reaches every timed leg, and the dumped arrays are the engine's results."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--contigs", "96", "--cpu-sample", "96"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "contigs/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "contigs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_dump_outputs_whole_and_sampled(tmp_path):
    import bench
    n, nl = 5000, 20000
    res = dict(call=(np.arange(n) % 3).astype(np.uint8), clade1=(3 * np.arange(n)).astype(np.int32),
               crit=0.5 * np.arange(n), member_off=np.arange(n + 1, dtype=np.int64),
               synteny=(np.arange(nl) % 2).astype(np.uint8), ann_winner=np.zeros((nl, 0), np.int32),
               call_counts=np.array([7, 8, 9], np.int64))
    bench.dump_outputs(res, str(tmp_path / "whole"))
    assert sorted(f.name for f in (tmp_path / "whole").iterdir()) == sorted(k + ".npy" for k in res if k != "ann_winner")
    for k, v in res.items():
        if k == "ann_winner":   # no elements: not written
            continue
        got = np.load(str(tmp_path / "whole" / (k + ".npy")))
        assert got.dtype == np.float64 and np.array_equal(got, v), k
    limit = 60000
    for d in ("a", "b"):
        written = bench.dump_outputs(res, str(tmp_path / d), limit=limit)
        assert written == sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= limit

    def load(d, k):
        return np.load(str(tmp_path / d / (k + ".npy")))
    for k in res:
        if k != "ann_winner":
            assert load("a", k).tobytes() == load("b", k).tobytes(), k   # the same sample every time
    assert np.array_equal(load("a", "call_counts"), [7, 8, 9])       # small arrays stay whole
    rows = load("a", "clade1") / 3
    assert 0 < len(rows) < n and np.all(np.diff(rows) > 0)
    assert np.array_equal(load("a", "crit") * 2, rows)               # per-contig arrays keep the same rows
    assert np.array_equal(load("a", "call"), rows % 3)


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_results(tmp_path):
    """--steps sets the step count of the resident and the strong-scaling leg; the dumped arrays equal the C restatement's
    results on the same seeded workload, and a second run with other step counts dumps the same bytes."""
    import bench
    from oracle import c_oracle
    contigs = 3000
    base = [sys.executable, os.path.join(ROOT, "bench.py"), "--contigs", str(contigs), "--no-stream"]
    runs = {"a": ["--steps", "3", "--warmup", "1", "--strong-contigs", "8000", "--cpu-sample", "64"],
            "b": ["--steps", "1", "--warmup", "0", "--no-strong", "--no-cpu-baseline"]}
    for d, extra in runs.items():
        out = subprocess.run(base + extra + ["--dump-outputs", str(tmp_path / d)], capture_output=True, text=True,
                             timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == int(extra[1]) and line["config"]["contigs_per_gpu"] == contigs
        if d == "a":
            assert line["strong"]["steps"] == 3 and line["parity"]["bit_exact"], line["parity"]
    _, batch, params, tax = bench.make_workload(bench.argparse.Namespace(workload="cfg2", contigs=contigs))
    full = c_oracle.score_batch(params, tax, batch)
    ref = {k: v for k, v in full.items() if v.size > 0}
    for d in runs:   # one file per non-empty result array, nothing else
        assert sorted(f.name for f in (tmp_path / d).iterdir()) == sorted(k + ".npy" for k in ref), d
    got = {k: np.load(str(tmp_path / "a" / (k + ".npy"))) for k in ref}
    assert all(got[k].shape == v.shape for k, v in ref.items())
    # arrays without elements are not dumped: the comparison takes them (empty) from the reference
    assert not helpers.compare_results(full, dict(full, **got), score_rtol=bench.SCORE_RTOL)
    for k in ref:
        assert got[k].tobytes() == np.load(str(tmp_path / "b" / (k + ".npy"))).tobytes(), k
