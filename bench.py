#!/usr/bin/env python3
"""bench.py — valid pairs/s through SAM -> pairs -> dedup -> 5 kb bins on N B200s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            our arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...   the reference's own CPU code (oracle/_ref), same workload
    python bench.py ... --dump-outputs DIR                    also write the last timed step's outputs as DIR/*.npy: the inputs
                                                              are seeded, so two builds can be compared output for output

Workload (BASELINE.json configs[1]): hg38 Micro-C 150-cycle stitched-read SAM ("flash" mode), 100 M read groups per
GPU, synthetic (microcket_b200/csrc/synth.h), sam2pairs + coordinate dedup + 5 kb binning.  One step = one pass of
that whole path over the GPU's shard.  `value` times the path with the SAM text already resident in HBM; `e2e` times
the same path through the host-buffer C-ABI calls (pinned host SAM in, pairs text + COO counts out).
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HG38 = ["chr1", "chr10", "chr11", "chr12", "chr13", "chr14", "chr15", "chr16", "chr17", "chr18", "chr19", "chr2", "chr20",
        "chr21", "chr22", "chr3", "chr4", "chr5", "chr6", "chr7", "chr8", "chr9", "chrM", "chrX", "chrY"]
HG38_LEN = [248956422, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616,
            242193529, 64444167, 46709983, 50818468, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717,
            16569, 156040895, 57227415]
MM10 = ["chr1", "chr10", "chr11", "chr12", "chr13", "chr14", "chr15", "chr16", "chr17", "chr18", "chr19", "chr2", "chr3", "chr4", "chr5",
        "chr6", "chr7", "chr8", "chr9", "chrM", "chrX", "chrY"]
MM10_LEN = [195471971, 130694993, 122082543, 120129022, 120421639, 124902244, 104043685, 98207768, 94987271, 90702639, 61431566,
            182113224, 160039680, 156508116, 151834684, 149736546, 145441459, 129401213, 124595110, 16299, 171031299, 91744698]
DEFAULT_RES = [2500000, 1000000, 500000, 250000, 100000, 50000, 25000, 10000, 5000]          # microcket:98
# --config: which BASELINE.json configuration the line measures.  The default line (what the driver records) is configs[1].
WORKLOADS = {
    "flash": {"mode": "flash", "genome": "hg38", "names": HG38, "lens": HG38_LEN, "chimeric": -1,
              "title": "BASELINE configs[1]: hg38 Micro-C 150-cycle stitched-read SAM (flash mode), sam2pairs + coordinate dedup + 5kb binning"},
    "unc": {"mode": "unc", "genome": "mm10", "names": MM10, "lens": MM10_LEN, "chimeric": 384,
            "title": "BASELINE configs[2]: mm10 Hi-C non-stitched paired reads (unc mode), 37.5 % chimeric / split alignments "
                     "(ligation 5'-end resolution, unc2pairs.h:191-308), sam2pairs + coordinate dedup + 5kb binning"},
    "multires": {"mode": "flash", "genome": "hg38", "names": HG38, "lens": HG38_LEN, "chimeric": -1,
                 "title": "BASELINE configs[4]: hg38 multi-resolution binning (2.5 Mb - 5 kb, cis + trans) of device-resident packed pairs to COO"},
}
WORKLOADS["krmdup"] = {"mode": "fastq", "genome": "hg38", "names": HG38, "lens": HG38_LEN, "chimeric": -1,
                       "title": "BASELINE configs[3] on one box: krmdup over interleaved paired-end FASTQ (2 x 16-base keys, first occurrence "
                                "wins, 20 % duplicated fragments), one sequencing lane per GPU (`-b`: inter-lane duplicates are retained, "
                                "microcket:428-451, so lanes are independent and need no collective)"}
WL = WORKLOADS["flash"]
RES = 5000
SEED = 0x4D4B0002
METRIC = "valid pairs/sec (SAM->dedup->binned)"
PART_RES = 5_000_000        # owner = hash(chr1, chr2, pos1 / 5 Mb): the least common multiple of the driver's default resolutions
                            # (microcket:98), so every duplicate and every cell of every resolution has exactly one owner
DUP_PER_1024 = 128          # 12.5 % of the read groups re-use the fragment of another group anywhere in the job (PCR duplicates
                            # with their own read ids, crossing shard boundaries): ~11 % of the pairs are removed by the dedup


DUMP_ROWS = 1 << 19         # --dump-outputs keeps at most this many rows of each array (a quarter of it for each of the nine COOs of
                            # --config multires): the largest dump (--config multires --sam) is 61.9 MB of .npy files


def synth_opts(mk, universe):
    return mk.synth_opts(dup_per_1024=DUP_PER_1024, dup_universe=universe, chimeric_per_1024=WL["chimeric"])


def dump_rows(torch, np, t, n, rows=None):
    """the first n rows of tensor t on the host: all of them when n <= rows (default DUMP_ROWS), else a sample drawn with the
    workload's seed (so the same n gives the same rows in every run and every build), in output order"""
    rows = rows or DUMP_ROWS
    idx = np.arange(n) if n <= rows else np.sort(np.random.default_rng(SEED).choice(n, rows, replace=False))
    return t[:n][torch.from_numpy(idx).to(t.device)].cpu().numpy()


def write_dump(d, np, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)
    print(f"[bench] --dump-outputs: {', '.join(f'{k}{list(v.shape)}' for k, v in arrays.items())} -> {d}", file=sys.stderr)


def dump_pipeline(d, torch, np, mk, pipe, n_pairs, kept, nnz, st, text_len):
    """--dump-outputs: what the last timed step handed its caller (rank 0's share when N > 1).  Integers as float64 (positions
    exceed float32's 24-bit mantissa), text bytes as float32."""
    kp = pipe.pairs if pipe.src_ptr == pipe.pairs.data_ptr() else pipe.kept_pairs(kept)
    rec = np.frombuffer(dump_rows(torch, np, kp.view(-1, 16), kept).tobytes(), dtype=mk.PAIR_DTYPE)
    coo_rows = DUMP_ROWS // 4 if pipe.multires else DUMP_ROWS
    coo = lambda a, b, c, z: np.stack([dump_rows(torch, np, x, z, coo_rows) for x in (a, b, c)], axis=1).astype(np.float64)
    arrays = {"counts": np.array([n_pairs, kept, nnz], dtype=np.float64),          # pairs emitted, pairs kept by the dedup, COO cells
              "s2p_log": np.array([getattr(st, f) for f in ("lowMap", "manyHits", "unpaired", "selfCircle", "trans", "cis10K", "cis1K", "cis0")],
                                  dtype=np.float64),
              f"coo_{RES}": coo(pipe.b1, pipe.b2, pipe.cnt, nnz),                    # bin1, bin2, count
              "kept_pairs": np.stack([rec[f].astype(np.float64) for f in mk.PAIR_DTYPE.names], axis=1),   # columns: PAIR_DTYPE's fields
              "pairs_text": dump_rows(torch, np, pipe.text, text_len).astype(np.float32)}
    if SAM_ON:
        arrays["sam_text"] = dump_rows(torch, np, pipe.samout, pipe.sam_len).astype(np.float32)
    if pipe.multires:                               # the other eight resolutions: their cell counts and their COOs
        cells = {r: c for r, c in pipe.multires_cells.items() if c is not None}
        arrays["multires_cells"] = np.array(sorted(cells.items()), dtype=np.float64)
        for r, (b1, b2, c) in pipe.mcoo.items():
            arrays[f"coo_{r}"] = coo(b1, b2, c, cells[r])
    write_dump(d, np, arrays)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def synth_to_device(torch, mk, first, count, device, universe):
    """→ (uint8 cuda tensor holding the SAM text, n_bytes)"""
    return mk.synth_device(torch, SEED, WL["mode"], WL["genome"], first, count, device=device, opts=synth_opts(mk, universe))


def reference_sample(torch, mk, n_groups, device, tmpdir, universe):
    """Write the first n_groups of the workload to a file for the CPU arm."""
    buf, nb = synth_to_device(torch, mk, 0, n_groups, device, universe)
    path = os.path.join(tmpdir, "sample.sam")
    host = buf[:nb].cpu().numpy()
    with open(path, "wb") as f:
        f.write(host.tobytes())
    del buf
    return path, nb


def cpu_pipeline_once(sam_path, tmpdir, threads):
    """reference sam2pairs (oracle/_ref, its own sources) -> oracle coordinate dedup + 5 kb binning.  → (pairs, seconds, kind)"""
    import oracle_lib
    ref = os.path.join(ROOT, "oracle", "_ref", "sam2pairs")
    pre = os.path.join(tmpdir, "cpu")
    t0 = time.time()
    if os.path.exists(ref):
        kind = "reference"
        out = subprocess.run([ref, sam_path, WL["mode"], pre, str(threads), "0.5", "10", "1" if SAM_ON else "0"], check=True, capture_output=True).stdout
    else:
        kind = "port"
        cli = os.path.join(ROOT, "oracle", "_build", "oracle_cli")
        if not os.path.exists(cli):
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "port"], check=True, capture_output=True)
        out = subprocess.run([cli, "sam2pairs", sam_path, WL["mode"], pre, str(threads), "0.5", "10", "1" if SAM_ON else "0"], check=True, capture_output=True).stdout
    orc = oracle_lib.load()
    pairs, n = orc.pairs_parse(out, WL["names"])
    keep, kept = orc.coord_dedup(pairs, n)
    orc.bin_coo(pairs, n, keep, WL["lens"], RES)
    return n, time.time() - t0, kind


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    """The reference's CPU implementation of the path on this box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    import microcket_b200 as mk
    threads = max(2, min(host_cores(), 8))          # the driver passes sthread = 8 (microcket:461-466); the program does not scale further
    sample_groups = args.cpu_groups
    tmpdir = tempfile.mkdtemp(prefix="mkbench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        path, nb = reference_sample(torch, mk, sample_groups, 0, tmpdir, args.groups * max(1, args.gpus))
        times, pairs, kind = [], 0, "reference"
        args.warmup = min(args.warmup, 1)              # one pass warms the page cache; every further pass costs ~30 s
        for it in range(args.warmup + args.steps):
            pairs, sec, kind = cpu_pipeline_once(path, tmpdir, threads)
            if it >= args.warmup:
                times.append(sec)
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    ms = 1e3 * sum(times) / len(times)
    val = pairs / (ms / 1e3)
    sample = f"{sample_groups} read groups ({nb / 1e9:.2f} GB SAM) of the same synthetic workload per step, page-cache-warm file in /dev/shm"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": dict(workload_config(args, max(1, args.gpus), args.groups), window_mb=args.window_mb,
                                                  reference_sample_read_groups=sample_groups),
            "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(args, world, groups):
    return {"workload": WL["title"], "sam_passthrough": "on (the driver's default, microcket:107)" if SAM_ON else "off",
            "dedup": ("seq: krmdup's rule (bases [5,21) of each mate, first occurrence wins, src/preprocess/krmdup.cpp) on the SAM's primary records, inside sam2pairs"
                      if DEDUP_SEQ else "coord: (lane, chr1,pos1,s1, chr2,pos2,s2) of the emitted pairs, same sort as the binning"),
            "read_groups_per_gpu": groups, "genome": WL["genome"], "mode": WL["mode"], "resolution": RES, "min_mapq": 10, "min_mapped_ratio": 0.5,
            "seed": SEED, "duplicates": f"{DUP_PER_1024}/1024 of the read groups copy the fragment of another group of the whole job (all shards)", "l2": "inputs (>= 60 GB of SAM text per step at full size) far exceed the 126 MB L2; no flush needed",
            "lanes": (f"{world} (one krmdup key table per GPU = `microcket -b`: duplicates across lanes are retained, microcket:428-451)" if DEDUP_SEQ else "1 (duplicates are removed across all shards)"),
            "parallelism": f"shard{world}: parse by read chunk, packed pairs to their owner hash(chr1,chr2,pos1/{PART_RES}) by the library's own NVLink peer-memory kernel (MICROCKET_XCHG=nccl: partition + NCCL all-to-all), dedup + COO owner-computes"}


class Pipeline:
    """The timed path on one rank: sam2pairs over the rank's resident shard -> (N > 1: owner partition + all-to-all) ->
    coordinate dedup + 5 kb binning with one sort.  Used by the timed loop and by the reduced-size verification."""

    def __init__(self, torch, mk, dist, groups, world, local, window_bytes):
        self.torch, self.mk, self.dist, self.world = torch, mk, dist, world
        dev = torch.device(f"cuda:{local}")
        self.cap_pairs = int(groups * (1.0 if world == 1 else 1.3)) + 4096
        self.text = torch.empty(groups * 96 + (1 << 20), dtype=torch.uint8, device=dev)
        self.pairs = torch.empty(self.cap_pairs * 16, dtype=torch.uint8, device=dev)
        self.ws = mk.PairsWorkspace(self.cap_pairs, device=local)
        self.recv = torch.empty(self.cap_pairs * 16, dtype=torch.uint8, device=dev) if world > 1 else None
        self.b1 = torch.empty(self.cap_pairs, dtype=torch.int32, device=dev); self.b2 = torch.empty_like(self.b1); self.cnt = torch.empty_like(self.b1)
        self.samout = torch.empty(int(groups * (1400 if WL["mode"] == "unc" else 800)) + (1 << 20), dtype=torch.uint8, device=dev) if SAM_ON else None
        self.s2p = mk.Sam2Pairs(mk.S2PConfig(mode=WL["mode"], threads=8, write_sam=SAM_ON, emit_text=True, emit_packed=True, device=local,
                                             window_bytes=window_bytes, sharded=(world > 1), rmdup=DEDUP_SEQ, rmdup_capacity=groups + 1024), WL["names"])
        self.sam_len = 0
        self.stream = torch.cuda.current_stream().cuda_stream
        self.src = self.pairs
        self.src_ptr = self.pairs.data_ptr()
        self.multires = False
        self.xchg_events = []
        # N > 1: the library's NVLink peer-memory exchange (csrc/xchg.cu); MICROCKET_XCHG=nccl: partition + NCCL all-to-all
        self.xchg = None
        if world > 1 and os.environ.get("MICROCKET_XCHG", "p2p") != "nccl":
            from microcket_b200 import shard
            self.xchg = mk.Xchg(world, dist.get_rank(), self.cap_pairs, device=local)
            shard.connect_xchg(torch, dist, self.xchg, dev)
            self.recv = None
            # every window's pairs are scattered on a side stream while the next window is parsed (MICROCKET_XCHG_OVERLAP=0: one scatter at the end)
            self.overlap = os.environ.get("MICROCKET_XCHG_OVERLAP", "1") != "0"
            if self.overlap:
                self.s2p.attach_xchg(self.xchg, PART_RES)

    def run(self, sam, nbytes, pair_events=None, text_len=None):
        torch = self.torch
        self.s2p.reset()
        io = self.s2p.run_device(sam.data_ptr(), nbytes, True, self.text.data_ptr(), self.text.numel(), self.pairs.data_ptr(), self.cap_pairs,
                                 d_sam=self.samout.data_ptr() if SAM_ON else 0, sam_cap=self.samout.numel() if SAM_ON else 0, stream=self.stream)
        n = io.n_pairs
        self.sam_len = io.sam_text_len
        if text_len is not None:
            text_len[0] = io.pairs_text_len
        src_ptr = self.pairs.data_ptr()
        if self.xchg is not None:
            xa, xb, xc = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            xa.record()
            if not self.overlap:
                self.xchg.scatter(self.pairs.data_ptr(), n, PART_RES, stream=self.stream)
            xb.record()
            src_ptr, n = self.xchg.finish(stream=self.stream)
            xc.record()
            self.xchg_events.append((xa, xb, xc))
        elif self.world > 1:
            from microcket_b200 import shard
            n, src = shard.exchange_pairs(self.mk, torch, self.dist, self.ws, self.pairs, n, self.recv, self.cap_pairs, PART_RES, self.stream)
            src_ptr = src.data_ptr()
        # duplicate removal and 5 kb binning share one sort (mk_pairs_dedup_bin_device)
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        if DEDUP_SEQ:                                  # duplicates are gone already (cfg.rmdup): binning only
            kept = n
            nnz = self.ws.bin(src_ptr, n, WL["lens"], RES, self.b1.data_ptr(), self.b2.data_ptr(), self.cnt.data_ptr(), self.cap_pairs, stream=self.stream)
        else:
            kept, nnz = self.ws.dedup_bin(src_ptr, n, WL["lens"], RES, self.b1.data_ptr(), self.b2.data_ptr(), self.cnt.data_ptr(), self.cap_pairs,
                                          stream=self.stream)
        eb.record()
        if pair_events is not None:
            pair_events.append((ea, eb, n))
        self.src_ptr = src_ptr
        if self.multires:
            self.run_multires(src_ptr, kept)
        return io.n_pairs, kept, nnz

    def run_multires(self, kept_ptr, kept):
        """the other eight default resolutions from the kept pairs: the five whose triangle fits HBM from ONE pass of the dense
        histogram (shared-memory diagonals), 50 / 25 / 10 kb through the sort path (5 kb came out of the dedup's own sort)"""
        torch = self.torch
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        self.hist.reset(stream=self.stream)
        self.hist.add(kept_ptr, kept, stream=self.stream)
        ev[1].record()
        cells = {RES: None}
        for k, r in enumerate(self.dense_res):
            b1, b2, c = self.mcoo[r]
            cells[r], _ = self.hist.coo(k, b1.data_ptr(), b2.data_ptr(), c.data_ptr(), b1.numel(), stream=self.stream)
        ev[2].record()
        for r in self.sparse_res:
            b1, b2, c = self.mcoo[r]
            cells[r] = self.ws.bin(kept_ptr, kept, WL["lens"], r, b1.data_ptr(), b2.data_ptr(), c.data_ptr(), b1.numel(), stream=self.stream)
        ev[3].record()
        self.multires_events.append(ev)
        self.multires_cells = cells

    def enable_multires(self):
        mk, torch = self.mk, self.torch
        self.multires = True
        self.dense_res = [r for r in DEFAULT_RES if r >= 100000]
        self.sparse_res = [r for r in DEFAULT_RES if r < 100000 and r != RES]
        self.hist = mk.Hist(WL["lens"], self.dense_res, device=self.b1.device.index)
        # COO buffers of their own per resolution (a dense one needs no more rows than its triangle has cells), so that a step
        # leaves all nine resolutions' counts behind, as a caller receives them
        rows = lambda r: min(self.cap_pairs, mk.Hist.cells(WL["lens"], r)[1])
        self.mcoo = {r: [torch.empty(rows(r), dtype=torch.int32, device=self.b1.device) for _ in range(3)] for r in self.dense_res + self.sparse_res}
        self.multires_events, self.multires_cells = [], {}

    def kept_pairs(self, kept):
        """the kept pairs of the last run as a uint8 cuda tensor (copied out of wherever the exchange left them)"""
        out = self.torch.empty(max(kept, 1) * 16, dtype=self.torch.uint8, device=self.b1.device)
        if kept:
            self.mk.lib().check_cuda_copy(out.data_ptr(), self.src_ptr, kept * 16)
        return out[:kept * 16]

    def close(self):
        self.s2p.close(); self.ws.close()
        if self.xchg is not None:
            self.xchg.close()


def verify_sharded(torch, mk, np, dist, args, world, rank, local):
    """Untimed and ASSERTED: the N-GPU path (shard by read chunk -> sam2pairs -> owner partition -> all-to-all -> dedup + binning
    per owner) at reduced size.  Every rank's kept pairs and COO triplets are gathered; rank 0 compares their union with (a) the
    CPU oracle (sam2pairs + coordinate dedup + binning over the whole input) and (b) the single-GPU path over the whole input."""
    import oracle_lib
    V = args.verify_groups
    universe = V * world
    dev = torch.device(f"cuda:{local}")
    sam, nb = synth_to_device(torch, mk, rank * V, V + (1 if rank + 1 < world else 0), local, universe)   # + the next shard's first group:
    pipe = Pipeline(torch, mk, dist, V + 1, world, local, 64 << 20)                                        # only the stream's last group is dropped
    n_pairs, kept, nnz = pipe.run(sam, nb)
    st = pipe.s2p.finish(0, 0)
    # gather (padded to the largest rank)
    sizes = torch.tensor([kept, nnz, n_pairs, int(st.groups)], dtype=torch.int64, device=dev)
    all_sizes = [torch.empty_like(sizes) for _ in range(world)]
    dist.all_gather(all_sizes, sizes)
    all_sizes = [x.tolist() for x in all_sizes]
    mk_, mz = max(x[0] for x in all_sizes), max(x[1] for x in all_sizes)
    kp = torch.zeros(mk_ * 16, dtype=torch.uint8, device=dev); kp[:kept * 16] = pipe.kept_pairs(kept)
    coo = torch.zeros(mz * 3, dtype=torch.int32, device=dev)
    coo[:nnz] = pipe.b1[:nnz]; coo[mz:mz + nnz] = pipe.b2[:nnz]; coo[2 * mz:2 * mz + nnz] = pipe.cnt[:nnz]
    kps = [torch.empty_like(kp) for _ in range(world)]; coos = [torch.empty_like(coo) for _ in range(world)]
    dist.all_gather(kps, kp); dist.all_gather(coos, coo)
    pipe.close()
    ok, why = True, ""
    if rank == 0:
        got_pairs = np.concatenate([np.frombuffer(kps[r][:all_sizes[r][0] * 16].cpu().numpy().tobytes(), dtype=mk.PAIR_DTYPE) for r in range(world)])
        got_coo = np.concatenate([np.stack([coos[r][k * mz:k * mz + all_sizes[r][1]].cpu().numpy().astype(np.uint32) for k in range(3)], axis=1)
                                  for r in range(world)])
        got_coo = got_coo[np.lexsort((got_coo[:, 1], got_coo[:, 0]))]
        key = lambda a: np.lexsort((a["strands"], a["pos2"], a["chr2"], a["pos1"], a["chr1"], a["lane"]))
        # (a) the CPU oracle on exactly what the ranks were given: one reference process per shard (each drops its stream's last
        # kept read group, pairutil.h:176 - the shards overlap by one group so that in all but rare cases nothing is lost), then
        # coordinate dedup + binning over the union of the shards' pairs
        orc = oracle_lib.load()
        texts, groups = [], 0
        if DEDUP_SEQ:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import sam_rmdup_oracle as RM
        for r in range(world):
            sh, nbs = synth_to_device(torch, mk, r * V, V + (1 if r + 1 < world else 0), local, universe)
            sam_r = sh[:nbs].cpu().numpy().tobytes()
            if DEDUP_SEQ:                          # one krmdup process per shard = per lane (`-b`: duplicates across lanes are retained, microcket:428-451)
                r1_r, _, _ = orc.krmdup(RM.sam_to_fastq(sam_r)[0])
                sam_r = RM.filter_sam(sam_r, RM.kept_runs(r1_r))
            op_r, _, ost_r = orc.sam2pairs(sam_r, WL["mode"], threads=8, write_sam=False)
            texts.append(op_r); groups += ost_r.groups
            del sh
        op = b"".join(texts)
        arr, n = orc.pairs_parse(op, WL["names"])
        if DEDUP_SEQ:
            keep, n_keep = None, n
            b1, b2, ct = orc.bin_coo(arr, n, None, WL["lens"], RES)
            exp = np.frombuffer(bytes(arr), dtype=mk.PAIR_DTYPE)[:n]
        else:
            keep, n_keep = orc.coord_dedup(arr, n)
            b1, b2, ct = orc.bin_coo(arr, n, keep, WL["lens"], RES)
            exp = np.frombuffer(bytes(arr), dtype=mk.PAIR_DTYPE)[:n][np.frombuffer(bytes(keep), dtype=np.uint8)[:n] == 1]
        checks = {"groups": sum(x[3] for x in all_sizes) == groups, "pairs": sum(x[2] for x in all_sizes) == n,
                  "kept": len(got_pairs) == n_keep and np.array_equal(got_pairs[key(got_pairs)], exp[key(exp)]),
                  "coo": got_coo[:, 0].tolist() == b1 and got_coo[:, 1].tolist() == b2 and got_coo[:, 2].tolist() == ct,
                  "duplicates_removed": (sum(x[3] for x in all_sizes) < 0.95 * universe) if DEDUP_SEQ else (n - n_keep > 0.05 * n)}
        if DEDUP_SEQ:                              # lanes are independent by definition: there is no unsharded result to compare with
            ok = all(checks.values()); why = json.dumps(checks)
            print(f"[bench] verified {world}-GPU path (--dedup seq, one lane per GPU) on {universe} read groups: {why}", file=sys.stderr)
        else:
            # (b) the single-GPU path over the whole input against the oracle over the whole input (one stream, one dropped group)
            sam1, nb1 = synth_to_device(torch, mk, 0, universe, local, universe)
            op1, _, ost1 = orc.sam2pairs(sam1[:nb1].cpu().numpy().tobytes(), WL["mode"], threads=8, write_sam=False)
            arr1, n1 = orc.pairs_parse(op1, WL["names"])
            keep1, n_keep1 = orc.coord_dedup(arr1, n1)
            c1, c2, cc = orc.bin_coo(arr1, n1, keep1, WL["lens"], RES)
            exp1 = np.frombuffer(bytes(arr1), dtype=mk.PAIR_DTYPE)[:n1][np.frombuffer(bytes(keep1), dtype=np.uint8)[:n1] == 1]
            one = Pipeline(torch, mk, None, universe, 1, local, 64 << 20)
            p1, k1, z1 = one.run(sam1, nb1)
            single = np.frombuffer(one.kept_pairs(k1).cpu().numpy().tobytes(), dtype=mk.PAIR_DTYPE)
            checks["single_gpu_equals_oracle"] = (p1 == n1 and k1 == n_keep1 and z1 == len(c1) and np.array_equal(single[key(single)], exp1[key(exp1)])
                                                  and one.cnt[:z1].cpu().numpy().astype(np.uint32).tolist() == cc)
            checks["sharded_vs_unsharded_kept_pairs_differ_by_at_most_world_minus_1"] = abs(len(got_pairs) - k1) <= world - 1
            one.close()
            ok = all(checks.values()); why = json.dumps(checks)
            print(f"[bench] verified {world}-GPU path on {universe} read groups: {why}", file=sys.stderr)
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
    dist.broadcast(flag, 0)
    if int(flag.item()) != 1:
        raise SystemExit(f"bench.py: the {world}-GPU result differs from the oracle / single-GPU result: {why}")
    VERIFY["result"] = {"read_groups": universe, "asserted": True,
                        "against": ("CPU oracle: one krmdup + sam2pairs replay per lane (shard), union binned; kept pairs + COO of all ranks gathered" if DEDUP_SEQ
                                    else "CPU oracle and single-GPU path, kept pairs + COO of all ranks gathered")}


def run_krmdup(args):
    """--config krmdup: FASTQ duplicate removal through the host C ABI (mk_dedup_push / pull from pinned host memory; there is no
    device-resident entry point for FASTQ, so `value` and `e2e` are the same measurement).  One lane per GPU, no collective.
    --impl reference: the reference's krmdup binary (oracle/_ref/krmdup, its own 4 + 1 threads) on a bounded sample file."""
    import torch
    import microcket_b200 as mk
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    P = args.groups if args.groups != 100_000_000 else 20_000_000             # read pairs per GPU (default 20 M = 11.9 GB of FASTQ)
    metric = "read pairs/sec (krmdup, interleaved FASTQ -> deduplicated FASTQ)"
    cfg = {"workload": WL["title"], "read_pairs_per_gpu": P, "key": "bases [5,21) of each mate (krmdup.cpp:231-234)", "seed": SEED,
           "l2": "inputs (>= 10 GB of FASTQ per step) far exceed the 126 MB L2; no flush needed", "parallelism": f"lane{world}: one lane per GPU, no exchange"}
    if args.impl == "reference":
        if rank != 0:
            return
        ref = os.path.join(ROOT, "oracle", "_ref", "krmdup")
        S = min(P, 5_000_000)
        tmpdir = tempfile.mkdtemp(prefix="mkbench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            src = os.path.join(tmpdir, "in.fq")
            with open(src, "wb") as f:
                for k in range(0, S, 1_000_000):
                    buf, nb = mk.synth_device(torch, SEED, "fastq", "hg38", k, min(1_000_000, S - k))
                    f.write(buf[:nb].cpu().numpy().tobytes())
            times = []
            kind = "reference" if os.path.exists(ref) else "port"
            for it in range(min(args.warmup, 1) + args.steps):
                for e in ("read1.fq", "read2.fq", "log"):
                    if os.path.exists(os.path.join(tmpdir, "o." + e)):
                        os.remove(os.path.join(tmpdir, "o." + e))
                t0 = time.time()
                if kind == "reference":
                    subprocess.run([ref, "-i", src, "-o", os.path.join(tmpdir, "o")], check=True, capture_output=True)
                else:
                    import oracle_lib
                    oracle_lib.load().krmdup(open(src, "rb").read())
                if it >= min(args.warmup, 1):
                    times.append(time.time() - t0)
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)
        ms = 1e3 * sum(times) / len(times)
        val = S / (ms / 1e3)
        print(json.dumps({"impl": "reference", "metric": metric, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": min(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "u8", "data": "synthetic", "config": dict(cfg, reference_sample_read_pairs=S),
                          "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": 5, "kind": kind,
                                           "sample": f"{S} read pairs per step, file in /dev/shm, files written"},
                          "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    mk.lib().require_gpu()
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")
    # this rank's lane: its own fragments (seed differs per lane), staged in pinned host memory
    parts, nb = [], 0
    for k in range(0, P, 2_000_000):
        buf, n = mk.synth_device(torch, SEED + 97 * rank, "fastq", "hg38", k, min(2_000_000, P - k), device=local)
        parts.append(buf[:n].cpu()); nb += n
    host = torch.empty(nb, dtype=torch.uint8).pin_memory()
    o = 0
    for t in parts:
        host[o:o + t.numel()] = t; o += t.numel()
    del parts
    out1 = torch.empty(nb // 2 + (1 << 20), dtype=torch.uint8).pin_memory(); out2 = torch.empty_like(out1).pin_memory()
    W = 256 << 20
    n1, n2 = C.c_size_t(), C.c_size_t()

    # one context: reset() between steps = a new krmdup process (empty key sets).  async_pull: a pull's device-to-host copies run while the
    # next push copies its window in; what a pull reported is in the host buffers once the next pull (or finish) has returned
    kd = mk.Krmdup(device=local, window_bytes=W, async_pull=os.environ.get("MICROCKET_KRMDUP_ASYNC", "1") != "0")

    def once():
        kd.reset()
        L = kd.lib.L
        a = b = 0
        off = 0
        while off < nb or off == 0:
            m = min(W, nb - off)
            kd.lib.check(L.mk_dedup_push(kd.h, C.cast(host.data_ptr() + off, C.c_char_p), m, int(off + m == nb)))
            off += m
            kd.lib.check(L.mk_dedup_pull(kd.h, out1.data_ptr() + a, out1.numel() - a, C.byref(n1), out2.data_ptr() + b, out2.numel() - b, C.byref(n2)))
            a += n1.value; b += n2.value                  # the buffers hold everything a window can produce: one pull per push
            if off >= nb:
                break
        stt = kd.finish()
        while True:                                       # nothing is left in practice; finish() again = the last copies have landed
            kd.lib.check(L.mk_dedup_pull(kd.h, out1.data_ptr() + a, out1.numel() - a, C.byref(n1), out2.data_ptr() + b, out2.numel() - b, C.byref(n2)))
            if n1.value == 0 and n2.value == 0:
                break
            a += n1.value; b += n2.value
        stt = kd.finish()
        return stt, a, b

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(min(args.warmup, 2)):
        once()
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        stt, n_out1, n_out2 = once()
    barrier()
    sec = (time.perf_counter() - t0) / args.steps
    clk = clocks.stop() if rank == 0 else None
    out_bytes = n_out1 + n_out2
    if args.dump_outputs and rank == 0:
        import numpy as np
        write_dump(args.dump_outputs, np, {"krmdup_log": np.array([stt.uniq, stt.dup, stt.discard], dtype=np.float64),
                                           "read1_fastq": dump_rows(torch, np, out1, n_out1).astype(np.float32),
                                           "read2_fastq": dump_rows(torch, np, out2, n_out2).astype(np.float32)})
    t = torch.tensor([sec, float(stt.pairs), float(nb), float(out_bytes), float(stt.uniq), float(stt.dup)], dtype=torch.float64, device=dev)
    if dist is not None:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        sec = float(tmax[0]); t = tsum
    if rank == 0:
        pairs, h2d, d2h = float(t[1]), float(t[2]), float(t[3])
        peak, peak_src = measured_peak()
        val = pairs / sec
        line = {"metric": metric, "value": val, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": min(args.warmup, 2),
                "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": dict(cfg, fastq_bytes_per_gpu=nb, uniq=float(t[4]), dup=float(t[5])),
                "roofline": {"bound": "hbm", "kernel": "krmdup path (host-streamed)", "achieved": (h2d + d2h) / sec / 1e9, "peak": peak * world, "unit": "GB/s",
                             "frac": (h2d + d2h) / sec / 1e9 / (peak * world), "traffic": None, "peak_source": peak_src,
                             "note": "B_dd = FASTQ bytes in + FASTQ bytes out (SURVEY 8d); the path is fed over PCIe, so this fraction is a PCIe figure, not a kernel figure"},
                "cpu_baseline": None,
                "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "api": "mk_dedup_push / mk_dedup_pull (cfg.async_pull) / mk_dedup_finish from pinned host buffers, wall clock incl. all copies, max over ranks"},
                "gpu_launches": None, "clocks": clk,
                "parity": "bit-exact against the reference krmdup binary (tests/test_gpu_krmdup.py, tests/test_gpu_cli.py)"}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


VERIFY = {}
SAM_ON = False
DEDUP_SEQ = False       # --dedup seq: SAM-space krmdup inside sam2pairs (cfg.rmdup) + binning, instead of coordinate dedup + binning


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--groups", type=int, default=int(os.environ.get("MK_BENCH_GROUPS", 100_000_000)), help="read groups per GPU")
    ap.add_argument("--e2e-groups", type=int, default=int(os.environ.get("MK_BENCH_E2E_GROUPS", 0)), help="read groups of the end-to-end leg (0 = --groups)")
    ap.add_argument("--cpu-groups", type=int, default=int(os.environ.get("MK_BENCH_CPU_GROUPS", 10_000_000)))
    ap.add_argument("--window-mb", type=int, default=int(os.environ.get("MK_BENCH_WINDOW_MB", 2040)))
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--config", default="flash", choices=sorted(WORKLOADS), help="BASELINE.json configuration (default: configs[1], the headline)")
    ap.add_argument("--sam", action="store_true", help="SAM passthrough on (sam2pairs argv[7]; the driver's default) in both arms")
    ap.add_argument("--dedup", default="coord", choices=["coord", "seq"],
                    help="coord: duplicates by (lane, chr1,pos1,s1, chr2,pos2,s2) of the emitted pairs, one sort with the binning (default; no reference "
                         "implementation exists). seq: the reference's own krmdup rule (2 x 16 read bases, src/preprocess/krmdup.cpp) applied to the "
                         "SAM's primary records before grouping - pinned by the reference binaries - then binning")
    ap.add_argument("--no-verify", action="store_true", help="skip the untimed, asserted reduced-size verification of the N-GPU path")
    ap.add_argument("--verify-groups", type=int, default=200_000, help="read groups per GPU of that verification")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                                                          "(float64 / float32, a seeded sample of at most %d rows per array, %d per COO "
                                                          "with --config multires)" % (DUMP_ROWS, DUMP_ROWS // 4))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs: it goes with --impl ours")
    global WL, SAM_ON, DEDUP_SEQ
    WL = WORKLOADS[args.config]; SAM_ON = args.sam; DEDUP_SEQ = args.dedup == "seq"
    if DEDUP_SEQ and args.config == "multires":
        raise SystemExit("bench.py: --dedup seq goes with --config flash / unc")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.config == "krmdup":
        return run_krmdup(args)
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import microcket_b200 as mk

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    mk.lib().require_gpu()                            # no CPU fallback
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")
    G = args.groups
    stream = torch.cuda.current_stream().cuda_stream

    # ---- resident workload
    universe = G * world
    if world > 1 and not args.no_verify:
        verify_sharded(torch, mk, np, dist, args, world, rank, local)      # raises (non-zero exit) when the N-GPU result is wrong
    sam, nbytes = synth_to_device(torch, mk, rank * G, G, local, universe)
    pipe = Pipeline(torch, mk, dist, G, world, local, args.window_mb << 20)
    s2p, ws, cnt = pipe.s2p, pipe.ws, pipe.cnt
    if args.config == "multires":
        pipe.enable_multires()

    def step():
        return pipe.run(sam, nbytes, pair_events, text_len)

    pair_events = []
    text_len = [0]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    pair_events.clear()
    if pipe.multires:
        pipe.multires_events.clear()
    s2p.enable_timing(True)
    clocks = ClockSampler(local)
    launches0 = s2p.launches() + ws.launches()
    kt0 = s2p.kernel_times()
    barrier()
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        n_pairs, kept, nnz = step()
    e1.record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    kt1 = s2p.kernel_times()
    launches = s2p.launches() + ws.launches() - launches0
    s2p.enable_timing(False)
    st = s2p.finish(0, 0) if world > 1 else s2p.finish()
    if args.dump_outputs and rank == 0:
        dump_pipeline(args.dump_outputs, torch, np, mk, pipe, n_pairs, kept, nnz, st, text_len[0])
    # size-independent properties of the last timed step, at full size (reported, not asserted: the parity tests are tests/):
    # every emitted pair is counted in exactly one class counter; the COO counts add up to the pairs kept by the dedup
    checks = None
    try:
        cls_sum = int(st.trans) + int(st.cis10K) + int(st.cis1K) + int(st.cis0)
        coo_sum = int(cnt[:int(nnz)].to(torch.int64).sum().item())
        checks = {"pairs_equal_class_counters": cls_sum == int(n_pairs), "coo_counts_sum_to_kept_pairs": coo_sum == int(kept),
                  "scope": "rank 0, last timed step"}
    except Exception as e:                                    # never let the report break the bench line
        checks = {"error": str(e)}
    t = torch.tensor([ms_total, float(n_pairs), float(kept), float(nnz)], dtype=torch.float64, device=dev)
    if dist is not None:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_total, n_pairs_all, kept_all, nnz_all = float(tmax[0]), float(tsum[1]), float(tsum[2]), float(tsum[3])
    else:
        n_pairs_all, kept_all, nnz_all = float(n_pairs), float(kept), float(nnz)
    ms_step = ms_total / args.steps
    value = n_pairs_all / (ms_step / 1e3)

    # ---- end to end through the host-buffer C ABI (pinned host SAM in; pairs text, kept pairs and COO out), every rank its shard
    e2e_res = None
    if not args.no_e2e:
        del sam
        pipe.text = pipe.pairs = pipe.recv = None
        torch.cuda.empty_cache()
        e2e_res = measure_e2e(torch, mk, np, dist, args, world, rank, local)

    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return

    io_text_len = text_len[0]
    # ---- roofline of the dominant kernel, from CUDA events recorded on the launching stream during the timed region
    peak, peak_src = measured_peak()
    dk = {k: (kt1[k][0] - kt0[k][0], kt1[k][1] - kt0[k][1]) for k in kt1}
    dom = max(dk, key=lambda k: dk[k][0])
    dom_ms, dom_n = dk[dom]
    lines = float(st.lines)                            # lines of one pass (reset() clears the stream totals each step)
    groups = float(st.groups)
    # Algorithmic bytes per step of every kernel (DESIGN.md section 3): what the kernel has to read and write, not what it
    # happens to move.  Only the newline scan touches every SAM byte; the parser needs the head of each line (the 112 bytes
    # it fetches cover QNAME..CIGAR), its newline offset and flag byte, and writes one 48-byte record per line (an upper
    # bound is avoided by counting one record per read group only); the group kernel reads those records and writes a
    # 32-byte result per group; emit reads the results and the read id (~40 B) and writes ~72 B of text + 16 B packed.
    text_b = float(io_text_len)                        # bytes of pair text of one pass
    alg = {"k_scan_chunks": nbytes + 4 * lines, "k_chunk_index": 8 * lines,
           "k_parse": 117.0 * lines + 48.0 * groups, "k_group": lines + 80.0 * groups,
           "k_emit": 32.0 * groups + (40.0 + 72.0 + 16.0) * n_pairs, "k_copy_sam": (2.0 * float(pipe.sam_len) + 9.0 * lines) if pipe.sam_len else 0.0,   # passthrough off: the launch only returns
           "k_rmdup": 136.0 * lines + 32.0 * groups}     # --dedup seq: 8 B of K2's notes + the two key windows' sectors (4 x 32 B) per line, one 16-byte table slot read + written per read pair
    per_kernel = {}
    for k, (ms_k, n_k) in dk.items():
        if ms_k > 0 and n_k > 0:
            gbs = alg[k] * args.steps / (ms_k / 1e3) / 1e9
            per_kernel[k] = {"ms_per_step": ms_k / args.steps, "launches_per_step": n_k / args.steps, "algorithmic_GBps": gbs, "frac": gbs / peak}
    alg_bytes_step = alg[dom]
    launches_per_step = max(1.0, dom_n / args.steps)
    achieved = (alg_bytes_step / launches_per_step) / (dom_ms / max(dom_n, 1) / 1e3) / 1e9 if dom_ms > 0 else 0.0
    stage_ms = sum(v[0] for v in dk.values()) / args.steps
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get(dom)
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "launches_per_step": launches_per_step, "avg_launch_ms": dom_ms / max(dom_n, 1),
                "algorithmic_bytes_per_launch": alg_bytes_step / launches_per_step,
                "s2p_stage": {"ms_per_step": stage_ms, "GBps": (nbytes + text_b + pipe.sam_len) / (stage_ms / 1e3) / 1e9 if stage_ms else 0.0,
                              "frac": ((nbytes + text_b + pipe.sam_len) / (stage_ms / 1e3) / 1e9 / peak) if stage_ms else 0.0,
                              "bytes": "SAM text in + pair text out + SAM passthrough written when on (SURVEY 8d B_s2p)"},
                "kernels": per_kernel}
    # the dedup + binning stage (pack, one radix sort of 16-byte records, unique/cell compaction), CUDA events around the call
    # on the launching stream: algorithmic = 16 B per pair in + 16 B per kept pair + 12 B per cell out; what the sort really
    # moves is 2 x 16 B per pair per executed pass (9 passes for the 69-bit key at 5 kb on hg38)
    try:
        torch.cuda.synchronize()
        p_ms = sum(a.elapsed_time(b) for a, b, _ in pair_events) / max(1, len(pair_events))
        p_n = sum(x for _, _, x in pair_events) / max(1, len(pair_events))
        alg_p = 16.0 * p_n + 16.0 * float(kept) + 12.0 * float(nnz)
        roofline["pairs_stage"] = {"ms_per_step": p_ms, "algorithmic_GBps": alg_p / (p_ms / 1e3) / 1e9, "frac": alg_p / (p_ms / 1e3) / 1e9 / peak,
                                   "radix_passes": 9, "implementation_GBps": (alg_p + 9 * 32.0 * p_n) / (p_ms / 1e3) / 1e9}
    except Exception as e:
        roofline["pairs_stage"] = {"error": str(e)}
    if pipe.xchg_events:
        ev = pipe.xchg_events[-args.steps:]
        roofline["exchange_stage"] = {"scatter_ms": sum(a.elapsed_time(b) for a, b, _ in ev) / len(ev),
                                      "wait_for_all_ranks_ms": sum(b.elapsed_time(c) for _, b, c in ev) / len(ev),
                                      "overlapped_with_parsing": bool(getattr(pipe, "overlap", False)),
                                      "scope": "rank 0; scatter = this rank's pairs written into their owners' HBM over NVLink, wait = until "
                                               "every rank's flag has arrived (includes the ranks' skew)"}

    # ---- end to end through the host-buffer C ABI (pinned host SAM in; pairs text, packed pairs and COO out)
    e2e = e2e_res
    # ---- reference CPU path beside it (bounded sample)
    cpu = None
    if not args.no_cpu and world == 1:
        tmpdir = tempfile.mkdtemp(prefix="mkbench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            path, nb = reference_sample(torch, mk, args.cpu_groups, local, tmpdir, universe)
            threads = max(2, min(host_cores(), 8))
            p, sec, kind = cpu_pipeline_once(path, tmpdir, threads)
            cpu = {"value": p / sec, "unit": "pairs/s", "cores": threads, "kind": kind, "host_cores": host_cores(), "passes": 1,   # not --steps: a pass takes tens of seconds
                   "sample": f"{args.cpu_groups} read groups ({nb / 1e9:.2f} GB SAM) of the same workload, one pass, {sec:.1f} s: "
                             f"reference sam2pairs (T={threads}) + oracle dedup/binning (1 thread)"}
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)

    line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": dict(workload_config(args, world, G), sam_bytes_per_gpu=nbytes, pairs_per_step=n_pairs_all, kept_after_dedup=kept_all,
                           coo_cells=nnz_all, window_mb=args.window_mb),
            "read_groups_per_s": universe / (ms_step / 1e3),     # input read groups of all ranks per second (SURVEY 8d asks for both rates)
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clk, "checks": checks,
            "parity": ("sam2pairs AND the duplicate removal pinned by the reference binaries (krmdup's own rule taken on the SAM, tests/test_gpu_s2p_rmdup.py); "
                       "binning UNPINNED (juicer_tools absent: checked against oracle/pairs_oracle.c + numpy only) - that stage is %.1f of the %.1f ms step"
                       if DEDUP_SEQ else
                       "sam2pairs pinned by the reference binary (tests/); coordinate dedup + binning UNPINNED (no reference implementation "
                       "exists: checked against oracle/pairs_oracle.c + numpy only) - that stage is %.1f of the %.1f ms step") % (
                          roofline.get("pairs_stage", {}).get("ms_per_step", 0.0), ms_step),
            "verify_sharded": VERIFY.get("result")}
    if pipe.multires:
        torch.cuda.synchronize()
        me = pipe.multires_events
        avg = lambda a, b: sum(e[a].elapsed_time(e[b]) for e in me) / max(1, len(me))
        line["multires"] = {"resolutions": DEFAULT_RES, "dense_histogram": pipe.dense_res, "sort_path": [RES] + pipe.sparse_res,
                            "hist_add_ms": avg(0, 1), "hist_coo_ms": avg(1, 2), "sort_bins_ms": avg(2, 3),
                            "cells_rank0": {str(k): v for k, v in pipe.multires_cells.items() if v is not None},
                            "hist_algorithmic_GBps": 16.0 * float(kept) / max(avg(0, 1), 1e-9) / 1e6,
                            "note": "N > 1: every resolution is owner-computed (partition at 5 Mb = lcm of the list), no reduce needed"}
        line["metric"] = "valid pairs/sec (SAM->dedup->binned at the nine default resolutions)"
    print(json.dumps(line))
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


def bind_near_gpu(local):
    """Pin this process to the host cores of the GPU's NUMA node (if any are in its affinity mask), so that the pinned staging
    buffers of the end-to-end leg are first-touched on the socket the GPU's PCIe root hangs off.  → description for the record"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        node = int(open(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node").read())
        if node < 0:
            return "numa node unknown"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        mine = os.sched_getaffinity(0) & cpus
        if not mine:
            return f"gpu on numa node {node}, none of this process's {len(os.sched_getaffinity(0))} cores there"
        os.sched_setaffinity(0, mine)
        return f"bound to {len(mine)} cores of numa node {node}"
    except Exception as e:                                    # never let this break the bench
        return f"not bound ({str(e)[:60]})"


def measure_e2e(torch, mk, np, dist, args, world, rank, local):
    """The same path through the host-buffer C ABI: pinned host SAM pushed window by window (H2D inside), pair text and packed
    pairs pulled to host memory (D2H inside), then duplicate removal + binning with the kept pairs and COO triplets brought back
    to the host.  N > 1: every rank streams its own shard and the packed pairs cross NVLink (owner partition + all-to-all)
    before the dedup.  Wall clock between barriers, max over ranks."""
    numa = bind_near_gpu(local)
    E = min(args.e2e_groups or args.groups, args.groups)
    if world > 1 and not args.e2e_groups:
        E = min(E, 30_000_000)                     # N ranks pin N x the shard in host memory: 20 GB per rank keeps an 8-GPU box within 160 GB
    dev = torch.device(f"cuda:{local}")
    host = out_text = out_pairs = None
    while True:                                    # the full-size leg needs ~75 GB of pinned host memory per rank: back off if the box cannot pin it
        try:
            sam_d, nb = synth_to_device(torch, mk, rank * E, E, local, E * world)
            host = torch.empty(nb, dtype=torch.uint8).pin_memory()
            host.copy_(sam_d[:nb])
            del sam_d
            torch.cuda.synchronize(); torch.cuda.empty_cache()
            out_text = torch.empty(E * 88 + (1 << 20), dtype=torch.uint8).pin_memory()
            out_pairs = torch.empty((E + 1024) * 16, dtype=torch.uint8).pin_memory()
            ok = 1
        except (RuntimeError, MemoryError) as e:
            print(f"[bench] e2e: cannot stage {E} read groups in pinned memory ({str(e)[:80]}); halving", file=sys.stderr)
            host = out_text = out_pairs = None
            ok = 0
        if dist is not None:                       # every rank runs the same size
            f = torch.tensor([ok], dtype=torch.int32, device=dev); dist.all_reduce(f, op=dist.ReduceOp.MIN); ok = int(f.item())
        if ok:
            break
        host = out_text = out_pairs = None
        E //= 2
        if E < 1_000_000:
            return {"error": "pinned host memory"}
    cap = int(E * (1.0 if world == 1 else 1.3)) + 4096
    ob1 = torch.empty(cap, dtype=torch.int32).pin_memory(); ob2 = torch.empty_like(ob1).pin_memory(); oc = torch.empty_like(ob1).pin_memory()
    ws = mk.PairsWorkspace(cap, device=local)
    W = 256 << 20
    s2p = mk.Sam2Pairs(mk.S2PConfig(mode=WL["mode"], threads=8, write_sam=False, emit_text=True, emit_packed=True, device=local, window_bytes=W,
                                    sharded=(world > 1), rmdup=DEDUP_SEQ, rmdup_capacity=E + 1024), WL["names"])
    if DEDUP_SEQ and world == 1:
        sd_pairs = torch.empty(cap * 16, dtype=torch.uint8, device=dev)
        sb1 = torch.empty(cap, dtype=torch.int32, device=dev); sb2 = torch.empty_like(sb1); sbc = torch.empty_like(sb1)
    if world > 1:
        from microcket_b200 import shard
        d_pairs = torch.empty(cap * 16, dtype=torch.uint8, device=dev); d_kept = torch.empty_like(d_pairs)
        db1 = torch.empty(cap, dtype=torch.int32, device=dev); db2 = torch.empty_like(db1); dbc = torch.empty_like(db1)
        kept_host = torch.empty(cap * 16, dtype=torch.uint8).pin_memory()
        stream = torch.cuda.current_stream().cuda_stream
        use_p2p = os.environ.get("MICROCKET_XCHG", "p2p") != "nccl"
        if use_p2p:
            xchg = mk.Xchg(world, rank, cap, device=local)
            shard.connect_xchg(torch, dist, xchg, dev)
    phases = {"stream_ms": 0.0, "drain_finish_ms": 0.0, "pairs_ms": 0.0}

    def once():
        t_a = time.perf_counter()
        s2p.reset()
        tl = pl = 0
        off = 0
        while off < nb:
            m = min(W, nb - off)
            s2p.push_ptr(host.data_ptr() + off, m, off + m == nb)
            off += m
            a, b = s2p.pull_into(out_text.data_ptr() + tl, out_text.numel() - tl, out_pairs.data_ptr() + pl * 16, E + 1024 - pl)
            tl += a; pl += b
        t_b = time.perf_counter()
        while True:
            a, b = s2p.pull_into(out_text.data_ptr() + tl, out_text.numel() - tl, out_pairs.data_ptr() + pl * 16, E + 1024 - pl)
            tl += a; pl += b
            if a == 0 and b == 0:
                break
        st = s2p.finish(0, 0) if world > 1 else s2p.finish()
        assert st.pairs == pl
        t_c = time.perf_counter()
        if DEDUP_SEQ and world == 1:                   # the pulled pairs are already deduplicated: back to the device for the binning, COO to the host
            sd_pairs[:pl * 16].copy_(out_pairs[:pl * 16], non_blocking=True)
            kept = pl
            nnz = ws.bin(sd_pairs.data_ptr(), pl, WL["lens"], RES, sb1.data_ptr(), sb2.data_ptr(), sbc.data_ptr(), cap, stream=torch.cuda.current_stream().cuda_stream)
            ob1[:nnz].copy_(sb1[:nnz], non_blocking=True); ob2[:nnz].copy_(sb2[:nnz], non_blocking=True); oc[:nnz].copy_(sbc[:nnz], non_blocking=True)
            torch.cuda.synchronize()
            moved = pl
        elif world == 1:
            kept, nnz = ws.dedup_bin_host(out_pairs.data_ptr(), pl, WL["lens"], RES, ob1.data_ptr(), ob2.data_ptr(), oc.data_ptr(), cap)
            moved = pl
        else:
            d_pairs[:pl * 16].copy_(out_pairs[:pl * 16], non_blocking=True)
            if use_p2p:
                xchg.scatter(d_pairs.data_ptr(), pl, PART_RES, stream=stream)
                src_ptr, n = xchg.finish(stream=stream)
            else:
                n, src = shard.exchange_pairs(mk, torch, dist, ws, d_pairs, pl, d_kept, cap, PART_RES, stream)
                src_ptr = src.data_ptr()
            if DEDUP_SEQ:                              # lanes: duplicates are gone (per lane), the owner only bins what it received
                kept = n
                nnz = ws.bin(src_ptr, n, WL["lens"], RES, db1.data_ptr(), db2.data_ptr(), dbc.data_ptr(), cap, stream=stream)
            else:
                kept, nnz = ws.dedup_bin(src_ptr, n, WL["lens"], RES, db1.data_ptr(), db2.data_ptr(), dbc.data_ptr(), cap, stream=stream)
            mk.lib().check_cuda_copy(d_kept.data_ptr(), src_ptr, kept * 16)
            kept_host[:kept * 16].copy_(d_kept[:kept * 16], non_blocking=True)
            ob1[:nnz].copy_(db1[:nnz], non_blocking=True); ob2[:nnz].copy_(db2[:nnz], non_blocking=True); oc[:nnz].copy_(dbc[:nnz], non_blocking=True)
            torch.cuda.synchronize()
            moved = pl
        t_d = time.perf_counter()
        phases["stream_ms"] += (t_b - t_a) * 1e3; phases["drain_finish_ms"] += (t_c - t_b) * 1e3; phases["pairs_ms"] += (t_d - t_c) * 1e3
        return pl, tl, kept, nnz, moved

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(2):
        once()
    for k in phases:
        phases[k] = 0.0
    reps = args.steps
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        pl, tl, kept, nnz, moved = once()
    barrier()
    sec = (time.perf_counter() - t0) / reps
    s2p.close(); ws.close()
    t = torch.tensor([sec, float(pl), float(nb + moved * 16), float(tl + pl * 16 + (0 if DEDUP_SEQ and world == 1 else kept * 16) + nnz * 12)], dtype=torch.float64, device=dev)
    if dist is not None:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        sec, pl_all, h2d, d2h = float(tmax[0]), float(tsum[1]), float(tsum[2]), float(tsum[3])
    else:
        pl_all, h2d, d2h = float(pl), float(t[2]), float(t[3])
    return {"value": pl_all / sec, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "read_groups_per_gpu": E, "host_numa": numa, "ms_per_step": sec * 1e3, "phases_ms_rank0": {k: v / reps for k, v in phases.items()},
            "api": "mk_s2p_push/pull/pull_packed/finish from pinned host buffers" +
                   (" (cfg.rmdup) + H2D of the packed pairs, mk_pairs_bin_device, D2H of the COO" if DEDUP_SEQ else " + mk_pairs_dedup_bin_host" if world == 1 else " + H2D of the packed pairs, mk_xchg_* exchange over NVLink, mk_pairs_dedup_bin_device, D2H of kept pairs and COO") +
                   "; wall clock incl. all copies, max over ranks"}


if __name__ == "__main__":
    main()
