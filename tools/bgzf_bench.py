"""BGZF inflate on the GPU (csrc/bgzf.cu) against host zlib, and `pairs2bins` on bgzipped input.

  python tools/bgzf_bench.py --out <record.json> [--pairs 20000000] [--reps 5]

Corpus: seeded .pairs text made on the GPU by the library's own sam2pairs path (synthetic unc-mode SAM over hg38), BGZF-compressed
by Python's zlib at levels 1, 6 and 9 in bgzip's 65 280-byte members (tests/bgzf_corpus.py, members compressed on all cores).
  inflate     mk_bgzf_inflate_device on device-resident input, CUDA events around the call (member table upload, kernel, error
              word read back), after warm-up; once over the whole file in one call, once in the ~4 100-member calls of a 256 MiB
              text chunk as pairs2bins makes them.  GB/s of output and of input, members per second.  Input and output are
              far larger than the 126 MB L2.
  host zlib   the same members inflated by zlib on every core of the host (a thread pool: zlib releases the GIL).
  pairs2bins  wall clock at the nine default resolutions (microcket:98) on the .pairs, the .pairs.gz and `gzip -dc | pairs2bins -`
              (files in a temporary directory; CUDA start-up included).
The card's name and power limit are read in the same run.
"""
import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bgzf_corpus as B  # noqa: E402
import microcket_b200 as mk  # noqa: E402
from norm_bench import DEFAULT_RES, HG38_LEN, card  # noqa: E402  (tools/ is on the path when run as a script)

HG38 = ["chr1", "chr10", "chr11", "chr12", "chr13", "chr14", "chr15", "chr16", "chr17", "chr18", "chr19", "chr2", "chr20", "chr21",
        "chr22", "chr3", "chr4", "chr5", "chr6", "chr7", "chr8", "chr9", "chrM", "chrX", "chrY"]


def pairs_text(torch, n_pairs, seed=5, window=2_000_000):
    """.pairs text of at least n_pairs pairs from the device sam2pairs path, in windows of read groups"""
    s2p = mk.Sam2Pairs(mk.S2PConfig(mode="unc", threads=8, emit_text=True), HG38)
    parts, pairs, first = [], 0, 0
    while pairs < n_pairs:
        buf, nb = mk.synth_device(torch, seed, "unc", "hg38", first, window)
        out = torch.empty(nb + 64, dtype=torch.uint8, device="cuda")
        io = s2p.run_device(buf.data_ptr(), nb, True, out.data_ptr(), nb)
        parts.append(out[:io.pairs_text_len].cpu().numpy().tobytes())
        pairs += io.n_pairs; first += window
        s2p.reset()
        del buf, out
    s2p.close()
    return b"".join(parts), pairs


def compress(text, level, pool):
    chunks = [text[p:p + B.BLOCK] for p in range(0, len(text), B.BLOCK)]
    return b"".join(pool.map(lambda c: B.member(c, level=level), chunks)) + B.EOF


def host_inflate(blob, mem, pool):
    import zlib

    def one(m):
        d0 = m.in_off + 18                                              # bgzip's header: XLEN 6
        return len(zlib.decompress(blob[d0:m.in_off + m.in_len - 8], -15))
    t0 = time.perf_counter()
    n = sum(pool.map(one, mem))
    return time.perf_counter() - t0, n


def gpu_inflate(torch, blob, mem, n_out, reps, per_call):
    d_in = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    out = torch.empty(n_out + 1, dtype=torch.uint8, device="cuda")
    calls = [mem[k:k + per_call] for k in range(0, len(mem), per_call)]
    bz = mk.Bgzf(max(len(c) for c in calls))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def once():
        for c in calls:
            bz.inflate(d_in.data_ptr(), c, out.data_ptr(), n_out)
    for _ in range(2):
        once()
    ms = []
    for _ in range(reps):
        e0.record(); once(); e1.record(); torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ok = out[:n_out].cpu().numpy().tobytes()
    bz.close()
    return sorted(ms), ok


def wall(cmd, reps=2):
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = subprocess.run(cmd, shell=True, capture_output=True)
        dt = time.perf_counter() - t0
        assert r.returncode == 0, r.stderr[-2000:]
        best = dt if best is None else min(best, dt)
    return best, r.stderr.decode().strip().splitlines()[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--pairs", type=int, default=20_000_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    mk.lib().require_gpu()
    rec = {"card": card(), "cpus": os.cpu_count(), "pairs": a.pairs, "levels": {}}
    text, n_pairs = pairs_text(torch, a.pairs)
    rec.update(pairs=n_pairs, text_bytes=len(text))
    pool = cf.ThreadPoolExecutor(os.cpu_count())
    tmp = tempfile.mkdtemp(prefix="bgzf_bench_")
    for level in (1, 6, 9):
        blob = compress(text, level, pool)
        mem, nb, n_out = mk.bgzf_scan(blob, cap=len(blob) // 28 + 1)
        assert nb == len(blob) and n_out == len(text)
        r = {"bytes_in": len(blob), "members": len(mem)}
        for name, per in (("one_call", len(mem)), ("chunk_calls", (256 << 20) // B.BLOCK)):
            ms, got = gpu_inflate(torch, blob, mem, n_out, a.reps, per)
            assert got == text, f"level {level}: the device inflate differs from the text"
            med = ms[len(ms) // 2]
            r[name] = {"calls": -(-len(mem) // per), "ms": ms, "out_GBps": n_out / med / 1e6, "in_GBps": len(blob) / med / 1e6,
                       "members_per_s": len(mem) / med * 1e3}
        hs = [host_inflate(blob, mem, pool) for _ in range(3)]
        t = min(h[0] for h in hs)
        assert hs[0][1] == n_out
        r["host_zlib"] = {"threads": os.cpu_count(), "s": t, "out_GBps": n_out / t / 1e9, "in_GBps": len(blob) / t / 1e9}
        if level == 6:
            open(os.path.join(tmp, "x.pairs"), "wb").write(text)
            open(os.path.join(tmp, "x.pairs.gz"), "wb").write(blob)
            open(os.path.join(tmp, "hg38.info"), "w").write("".join(f"{n}\t{l}\n" for n, l in zip(HG38, HG38_LEN)))
            exe, res = os.path.join(os.path.dirname(mk.LIB_PATH), "bin", "pairs2bins"), ",".join(map(str, DEFAULT_RES))
            info = os.path.join(tmp, "hg38.info")
            cmds = {"pairs": f"{exe} -r {res} {tmp}/x.pairs {tmp}/a {info}",
                    "pairs_gz": f"{exe} -r {res} {tmp}/x.pairs.gz {tmp}/b {info}",
                    "gzip_dc_pipe": f"gzip -dc {tmp}/x.pairs.gz | {exe} -r {res} - {tmp}/c {info}"}
            r["pairs2bins_s"] = {k: wall(c) for k, c in cmds.items()}
            for k in ("b", "c"):
                for q in DEFAULT_RES:
                    assert open(f"{tmp}/a.{q}.coo", "rb").read() == open(f"{tmp}/{k}.{q}.coo", "rb").read()
        rec["levels"][str(level)] = r
        print(level, json.dumps(r)[:600], flush=True)
    subprocess.run(["rm", "-rf", tmp])
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(rec, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
