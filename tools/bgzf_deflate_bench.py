"""BGZF deflate on the GPU (csrc/bgzf_deflate.cu) against host zlib, and `bgzip` on a file.

  python tools/bgzf_deflate_bench.py --out <record.json> [--pairs 20000000] [--reps 5]

Corpus: the one tools/bgzf_bench.py inflates: seeded .pairs text made on the GPU by the library's own sam2pairs path (synthetic
unc-mode SAM over hg38), cut in bgzip's 65 280-byte members.
  kernel      mk_bgzf_deflate_device on device-resident input, CUDA events around the call (kernels, size read-back), after
              warm-up; once over the whole text in one call, once in 256 MiB calls as `bgzip` makes them.  GB/s of input,
              members per second.  Input and output are far larger than the 126 MB L2.
  size        compressed bytes against zlib levels 1 and 6 on the same members (bgzip's header and trailer included).
  host zlib   the same members compressed by zlib at levels 1 and 6 on every core of the host (a thread pool: zlib releases
              the GIL).
  bgzip       wall clock of `bgzip -k -f` on the text file (CUDA start-up included), and of `bgzip -d -c`.
  round trips the output inflated by host zlib and by mk_bgzf_inflate_device equals the text; `pairs2bins` on the bgzip output
              writes the same .coo files as on the plain text.
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
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bgzf_corpus as B  # noqa: E402
import microcket_b200 as mk  # noqa: E402
from bgzf_bench import HG38, host_inflate, pairs_text, wall  # noqa: E402  (tools/ is on the path when run as a script)
from norm_bench import DEFAULT_RES, HG38_LEN, card  # noqa: E402


def gpu_deflate(torch, text, reps, per_call):
    d_in = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    cap = mk.bgzf_deflate_bound(len(text))
    out = torch.empty(cap + 1, dtype=torch.uint8, device="cuda")
    calls = [(p, min(per_call, len(text) - p)) for p in range(0, len(text), per_call)]
    bd = mk.BgzfDeflate(max(n for _, n in calls))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def once():
        o = 0
        for p, n in calls:
            k, _ = bd.deflate(d_in.data_ptr() + p, n, out.data_ptr() + o, cap - o)
            o += k
        return o
    for _ in range(2):
        once()
    ms = []
    for _ in range(reps):
        e0.record(); n_out = once(); e1.record(); torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    blob = out[:n_out].cpu().numpy().tobytes()
    bd.close()
    return sorted(ms), blob


def host_deflate(text, level, pool):
    chunks = [text[p:p + B.BLOCK] for p in range(0, len(text), B.BLOCK)]
    t0 = time.perf_counter()
    n = sum(pool.map(lambda c: len(B.member(c, level=level)), chunks))
    return time.perf_counter() - t0, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--pairs", type=int, default=20_000_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    mk.lib().require_gpu()
    rec = {"card": card(), "cpus": os.cpu_count(), "pairs": a.pairs}
    text, n_pairs = pairs_text(torch, a.pairs)
    rec.update(pairs=n_pairs, text_bytes=len(text), members=-(-len(text) // B.BLOCK))
    pool = cf.ThreadPoolExecutor(os.cpu_count())
    blob = None
    for name, per in (("one_call", len(text)), ("calls_256MiB", (256 << 20) // B.BLOCK * B.BLOCK)):
        ms, got = gpu_deflate(torch, text, a.reps, per)
        assert blob is None or got == blob, "the bytes depend on the call cut"
        blob = got
        med = ms[len(ms) // 2]
        rec[name] = {"calls": -(-len(text) // per), "ms": ms, "in_GBps": len(text) / med / 1e6, "out_GBps": len(blob) / med / 1e6,
                     "members_per_s": rec["members"] / med * 1e3}
        print(name, json.dumps(rec[name]), flush=True)
    rec["bytes"] = {"gpu": len(blob), "ratio_gpu": len(text) / len(blob)}
    for level in (1, 6):
        ts = [host_deflate(text, level, pool) for _ in range(2)]
        t, n = min(x[0] for x in ts), ts[0][1]
        rec["bytes"][f"zlib{level}"] = n
        rec["bytes"][f"ratio_zlib{level}"] = len(text) / n
        rec[f"host_zlib{level}"] = {"threads": os.cpu_count(), "s": t, "in_GBps": len(text) / t / 1e9}
    rec["kernel_over_host_zlib6"] = rec["one_call"]["in_GBps"] / rec["host_zlib6"]["in_GBps"]
    print(json.dumps(rec["bytes"]), flush=True)
    # round trips
    mem, nb, n_out = mk.bgzf_scan(blob, cap=rec["members"] + 1)
    assert nb == len(blob) and n_out == len(text) and len(mem) == rec["members"]
    assert host_inflate(blob, mem, pool)[1] == len(text)
    assert b"".join(pool.map(lambda m: zlib.decompress(blob[m.in_off + 18:m.in_off + m.in_len - 8], -15), mem)) == text
    assert mk.bgzf_decompress(blob) == text
    rec["round_trips"] = {"host_zlib": True, "mk_bgzf_inflate_device": True}
    tmp = tempfile.mkdtemp(prefix="bgzf_deflate_bench_")
    bin_dir = os.path.join(os.path.dirname(mk.LIB_PATH), "bin")
    open(os.path.join(tmp, "x.pairs"), "wb").write(text)
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        r = subprocess.run([f"{bin_dir}/bgzip", "-k", "-f", f"{tmp}/x.pairs"], capture_output=True)
        dt = time.perf_counter() - t0
        assert r.returncode == 0, r.stderr[-2000:]
        best = dt if best is None else min(best, dt)
    assert open(f"{tmp}/x.pairs.gz", "rb").read() == blob + B.EOF, "bgzip differs from the library call"
    t0 = time.perf_counter()
    r = subprocess.run(f"{bin_dir}/bgzip -d -c {tmp}/x.pairs.gz > {tmp}/y.pairs", shell=True, capture_output=True)
    dts = time.perf_counter() - t0
    assert r.returncode == 0 and open(f"{tmp}/y.pairs", "rb").read() == text
    rec["bgzip_s"] = {"compress_file": best, "compress_in_GBps": len(text) / best / 1e9, "decompress_file": dts,
                      "host_zlib6_all_cores": rec["host_zlib6"]["s"], "host_zlib1_all_cores": rec["host_zlib1"]["s"]}
    open(os.path.join(tmp, "hg38.info"), "w").write("".join(f"{n}\t{ln}\n" for n, ln in zip(HG38, HG38_LEN)))
    exe, res, info = os.path.join(bin_dir, "pairs2bins"), ",".join(map(str, DEFAULT_RES)), os.path.join(tmp, "hg38.info")
    wall(f"{exe} -r {res} {tmp}/x.pairs {tmp}/a {info}", reps=1)
    wall(f"{exe} -r {res} {tmp}/x.pairs.gz {tmp}/b {info}", reps=1)
    for q in DEFAULT_RES:
        assert open(f"{tmp}/a.{q}.coo", "rb").read() == open(f"{tmp}/b.{q}.coo", "rb").read()
    rec["round_trips"]["pairs2bins_coo_equal"] = True
    print(json.dumps(rec["bgzip_s"]), flush=True)
    subprocess.run(["rm", "-rf", tmp])
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(rec, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
