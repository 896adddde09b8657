"""bench.py --dump-outputs: at a size where nothing is sampled the dumped outputs of the last timed step are the CPU oracle's, two
runs dump the same arrays whatever --steps is, --steps timed steps really run, and a sampled dump holds the seeded subset of
the full output's rows in output order."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import microcket_b200 as mk
from oracle_lib import sort_pairs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

G = 5000                        # read groups: every output stays below the rows a dump keeps


def load(out):
    arrays = {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out)) < 64 << 20
    return arrays


def run_bench(out, steps, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--no-cpu",
                        "--no-e2e", "--dump-outputs", str(out), *args], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return line, load(out)


def oracle_outputs(oracle, torch):
    buf, nb = mk.synth_device(torch, bench.SEED, "flash", "hg38", 0, G,
                              opts=mk.synth_opts(dup_per_1024=bench.DUP_PER_1024, dup_universe=G, chimeric_per_1024=-1))
    op, _, ost = oracle.sam2pairs(buf[:nb].cpu().numpy().tobytes(), "flash", threads=8, write_sam=False)
    arr, n = oracle.pairs_parse(op, bench.HG38)
    keep, kept = oracle.coord_dedup(arr, n)
    return op, ost, arr, n, keep, kept


def test_flash_dump_is_the_oracles_and_steps_run(tmp_path, oracle):
    import torch
    l1, a = run_bench(tmp_path / "a", 1, "--groups", str(G))
    l3, b = run_bench(tmp_path / "b", 3, "--groups", str(G))
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert l3["gpu_launches"] == 3 * l1["gpu_launches"] > 0           # every timed step launches the same kernels

    op, ost, arr, n, keep, kept = oracle_outputs(oracle, torch)
    b1, b2, ct = oracle.bin_coo(arr, n, keep, bench.HG38_LEN, bench.RES)
    assert a["counts"].tolist() == [n, kept, len(ct)] and kept < n
    assert a["s2p_log"].tolist() == [int(x.split(b"\t")[1]) for x in ost.log_text().splitlines()]
    assert a["coo_5000"].tolist() == [list(r) for r in zip(b1, b2, ct)]
    exp = np.frombuffer(bytes(arr), dtype=mk.PAIR_DTYPE)[:n][np.frombuffer(bytes(keep), dtype=np.uint8)[:n] == 1]
    exp = np.stack([exp[f].astype(np.float64) for f in mk.PAIR_DTYPE.names], axis=1)
    order = lambda x: x[np.lexsort(x.T[::-1])]
    assert np.array_equal(order(a["kept_pairs"]), order(exp))
    assert sort_pairs(a["pairs_text"].astype(np.uint8).tobytes()) == sort_pairs(op)


def test_multires_dump_holds_every_resolution_and_samples_by_seed(tmp_path, oracle, monkeypatch, capsys):
    """all nine COOs against the oracle; then the same run in this process with DUMP_ROWS cut to 1000, so that every long array
    is sampled: each dumped array must be the full one's rows at the seeded indices"""
    import torch
    _, full = run_bench(tmp_path / "full", 2, "--config", "multires", "--groups", str(G))
    _, _, arr, n, keep, kept = oracle_outputs(oracle, torch)
    assert full["multires_cells"][:, 0].tolist() == sorted(r for r in bench.DEFAULT_RES if r != bench.RES)
    for r in bench.DEFAULT_RES:
        b1, b2, ct = oracle.bin_coo(arr, n, keep, bench.HG38_LEN, r)
        assert full[f"coo_{r}"].tolist() == [list(x) for x in zip(b1, b2, ct)], r

    rows = 1000
    monkeypatch.setattr(bench, "DUMP_ROWS", rows)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", "2", "--warmup", "1", "--no-cpu", "--no-e2e", "--config",
                                      "multires", "--groups", str(G), "--dump-outputs", str(tmp_path / "sampled")])
    bench.main()
    capsys.readouterr()
    sampled = load(tmp_path / "sampled")
    assert sampled.keys() == full.keys()
    n_sampled = 0
    for k, a in full.items():
        cap = rows // 4 if k.startswith("coo_") else rows
        if len(a) <= cap:
            assert np.array_equal(sampled[k], a), k
            continue
        idx = np.sort(np.random.default_rng(bench.SEED).choice(len(a), cap, replace=False))
        assert np.array_equal(sampled[k], a[idx]), k
        n_sampled += 1
    assert n_sampled >= 4                      # kept pairs, pairs text and the finer COOs
