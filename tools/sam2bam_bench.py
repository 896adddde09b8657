"""`sam2bam` (coordinate-sorted BAM + .bai on the GPU, csrc/bam_out.cu) on SAM of the size a user runs.

  python tools/sam2bam_bench.py --out <record.json> [--groups 10000000] [--reps 2] [--dir /dev/shm]

Input: hg38 flash-mode SAM made on the GPU by mk_synth_device (seeded), with an @SQ header from the genome table, written to
--dir (/dev/shm when it is writable: the input is read from memory, so the wall clock is the tool's and not the disk's).
  wall        `sam2bam -o x.bam in.sam` in core, and with MICROCKET_SORT_MB set to a fifth of the input so that it spills
              about five runs and merges them; best of --reps, CUDA start-up included; GB/s of SAM input.  The two outputs
              must be the same bytes.
  splits      the library calls on one device-resident piece of the same SAM (--split-groups read groups), CUDA events
              around each phase: encode (line index, sizes, records), sort + gather (keys, radix sort, gather in 256 MiB
              windows), deflate (mk_bgzf_deflate_device on those windows), index (per-record bins, linear index, chunk runs)
              and the .bai layout.
The card's name and power limit are read in the same run.  No samtools comparison is made: samtools is not in this image.
"""
import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import microcket_b200 as mk  # noqa: E402
from norm_bench import card  # noqa: E402  (tools/ is on the path when run as a script)

HG38 = list(zip(["chr1", "chr10", "chr11", "chr12", "chr13", "chr14", "chr15", "chr16", "chr17", "chr18", "chr19", "chr2", "chr20", "chr21",
                 "chr22", "chr3", "chr4", "chr5", "chr6", "chr7", "chr8", "chr9", "chrM", "chrX", "chrY"],
                [248956422, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616,
                 242193529, 64444167, 46709983, 50818468, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717,
                 16569, 156040895, 57227415]))
SAM2BAM = os.path.join(os.path.dirname(mk.LIB_PATH), "bin", "sam2bam")
MB = 1 << 20


def write_sam(torch, path, groups, piece=1000000):
    with open(path, "wb") as f:
        f.write("".join(f"@SQ\tSN:{n}\tLN:{l}\n" for n, l in HG38).encode())
        for first in range(0, groups, piece):
            buf, n = mk.synth_device(torch, 21, "flash", "hg38", first, min(piece, groups - first))
            f.write(buf[:n].cpu().numpy().tobytes())
    return os.path.getsize(path)


def wall(args, env, reps):
    best, err = None, ""
    for _ in range(reps):
        t0 = time.perf_counter()
        r = subprocess.run(args, capture_output=True, env=dict(os.environ, **env))
        dt = time.perf_counter() - t0
        assert r.returncode == 0, r.stderr[-2000:]
        best, err = (dt if best is None else min(best, dt)), r.stderr.decode().strip().splitlines()[-1]
    return best, err


def splits(torch, groups):
    """CUDA-event times of the library's phases on one device-resident piece of flash SAM"""
    buf, n = mk.synth_device(torch, 22, "flash", "hg38", 0, groups)
    win = 256 * MB
    bam = mk.Bam(HG38, n + 16, groups * 4 + 16)
    bd = mk.BgzfDeflate(win + 65280)
    rec = torch.empty(2 * n + 1024, dtype=torch.uint8, device="cuda")
    off = torch.empty(groups * 4 + 16, dtype=torch.int64, device="cuda")
    out = torch.empty(2 * win + 4 * 65280, dtype=torch.uint8, device="cuda")
    z = torch.empty(mk.bgzf_deflate_bound(2 * win + 4 * 65280), dtype=torch.uint8, device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def once():
        t = {"encode": 0.0, "sort_gather": 0.0, "deflate": 0.0, "index": 0.0}
        a, b = ev(), ev()
        a.record(); nr, rb = bam.encode(buf.data_ptr(), n, rec.data_ptr(), rec.numel(), off.data_ptr()); b.record(); b.synchronize()
        t["encode"] += a.elapsed_time(b)
        a.record(); bam.sort(rec.data_ptr(), off.data_ptr(), nr); b.record(); b.synchronize()
        t["sort_gather"] += a.elapsed_time(b)
        bam.index_reset()
        i0, u, zb, coff = 0, 0, 0, []
        while i0 < nr:
            a.record(); i1, nb, d_off = bam.gather(i0, win, out.data_ptr(), out.numel()); b.record(); b.synchronize()
            t["sort_gather"] += a.elapsed_time(b)
            a.record(); bam.index_add(out.data_ptr(), d_off, i1 - i0, u); b.record(); b.synchronize()
            t["index"] += a.elapsed_time(b)
            a.record(); k, mem = bd.deflate(out.data_ptr(), nb, z.data_ptr(), z.numel()); b.record(); b.synchronize()
            t["deflate"] += a.elapsed_time(b)
            coff += [zb + m.in_off for m in mem]
            zb += k; u += nb; i0 = i1
        t0 = time.perf_counter(); bai = bam.bai(coff + [zb]); t["bai_layout_host"] = (time.perf_counter() - t0) * 1e3
        return t, nr, rb, zb, len(bai)
    once()
    runs = [once() for _ in range(3)]
    t = {k: min(r[0][k] for r in runs) for k in runs[0][0]}
    _, nr, rb, zb, nbai = runs[0]
    bam.close(); bd.close()
    return {"sam_bytes": n, "records": nr, "record_bytes": rb, "bgzf_bytes": zb, "bai_bytes": nbai,
            "ms": {k: round(v, 2) for k, v in t.items()},
            "sam_GBps": {k: round(n / (v * 1e6), 2) for k, v in t.items() if v > 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--groups", type=int, default=10000000)
    ap.add_argument("--split-groups", type=int, default=1500000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--dir", default="/dev/shm" if os.access("/dev/shm", os.W_OK) else None)
    a = ap.parse_args()
    import torch
    mk.lib().require_gpu()
    rec = {"card": card(), "groups": a.groups}
    with tempfile.TemporaryDirectory(dir=a.dir) as d:
        sam = os.path.join(d, "in.sam")
        t0 = time.perf_counter()
        size = write_sam(torch, sam, a.groups)
        rec["input"] = {"sam_bytes": size, "dir": a.dir or tempfile.gettempdir(), "write_s": round(time.perf_counter() - t0, 2)}
        s_core, info_core = wall([SAM2BAM, "-o", os.path.join(d, "a.bam"), sam], {}, a.reps)
        sort_mb = max(1024, size // 5 // MB)
        s_spill, info_spill = wall([SAM2BAM, "-o", os.path.join(d, "b.bam"), sam], {"MICROCKET_SORT_MB": str(sort_mb)}, a.reps)
        same = filecmp.cmp(os.path.join(d, "a.bam"), os.path.join(d, "b.bam"), shallow=False) and \
            filecmp.cmp(os.path.join(d, "a.bam.bai"), os.path.join(d, "b.bam.bai"), shallow=False)
        rec["wall"] = {
            "in_core": {"s": round(s_core, 3), "sam_GBps": round(size / s_core / 1e9, 2), "info": info_core},
            "spill": {"sort_mb": sort_mb, "s": round(s_spill, 3), "sam_GBps": round(size / s_spill / 1e9, 2), "info": info_spill},
            "bam_bytes": os.path.getsize(os.path.join(d, "a.bam")), "spill_output_identical": same}
    rec["splits"] = splits(torch, a.split_groups)
    rec["samtools"] = "not measured (samtools is not in this image)"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
