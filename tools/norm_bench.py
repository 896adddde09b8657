"""Matrix balancing on the GPU (csrc/norm.cu): time, products and bytes per product of VC, VC_SQRT and KR (per chromosome) and of
GW_VC / GW_KR (whole-genome matrix) and INTER_VC / INTER_KR (inter-chromosomal entries) at the nine default resolutions
(microcket:98), on seeded synthetic pairs over hg38 (power-law distance decay p(d) ~ 1/d, a trans fraction) binned on the GPU;
plus an independent scipy `bnewt` on the 100 kb matrices of the largest size (every chromosome's, and the genome-wide one) as
the CPU reference points.

  python tools/norm_bench.py --out <record.json> [--pairs 20000000,250000000]

Bytes per product are algorithmic: 8 B per stored entry (u32 column + u32 count; both halves of the symmetric matrix of the
scope, the diagonal once: 2 nnz - diagonal) + 8 B per row pointer + 8 B per row of y.  The input vector u (8 B per bin, 4.9 MB at 5 kb) is a gather that
stays in L2 and is not counted.  The rate is compared with the HBM peak bench.py uses (MEASURED_PEAKS.json `hbm_gbs`, else
bench.py's fallback; the record names which).
The full products are the row sums and the sum factors (every row); KR's products skip the rows of chromosomes that are done.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HG38_LEN = [248956422, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616,
            242193529, 64444167, 46709983, 50818468, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717,
            16569, 156040895, 57227415]
DEFAULT_RES = [2500000, 1000000, 500000, 250000, 100000, 50000, 25000, 10000, 5000]    # microcket:98


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def synth_pairs(torch, n, seed, trans=0.2):
    """mk_pair records (16 B) on the device: chromosome by length, 20 % trans, intra distance log-uniform in [1, length)"""
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    L = torch.tensor(HG38_LEN, dtype=torch.float64, device="cuda")
    cdf = torch.cumsum(L / L.sum(), 0)
    c1 = torch.clamp(torch.searchsorted(cdf, torch.rand(n, generator=g, device="cuda", dtype=torch.float64)), max=len(HG38_LEN) - 1)
    c2 = torch.where(torch.rand(n, generator=g, device="cuda") < trans, torch.randint(0, len(HG38_LEN), (n,), generator=g, device="cuda"), c1)
    p1 = (torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * (L[c1] - 1)).long() + 1
    d = torch.exp(torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * torch.log(L[c1])).long()
    sign = torch.where(torch.rand(n, generator=g, device="cuda") < 0.5, -1, 1)
    Lc2 = L[c2].long()
    p2 = torch.where(c1 == c2, torch.minimum(torch.clamp(p1 + sign * d, min=1), Lc2),
                     (torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * (L[c2] - 1)).long() + 1)
    del d, sign, Lc2
    sw = c1 > c2
    rec = torch.zeros((n, 4), dtype=torch.int32, device="cuda")
    rec[:, 0] = torch.where(sw, p2, p1).int(); rec[:, 1] = torch.where(sw, p1, p2).int()
    rec[:, 2] = (torch.minimum(c1, c2) | (torch.maximum(c1, c2) << 16)).int()
    return rec


def matrix_shape(torch, b1, b2, nnz, res, scope="INTRA"):
    off = torch.tensor(np.cumsum([l // res + 1 for l in HG38_LEN]), dtype=torch.int64, device="cuda")
    x, y = b1[:nnz].long(), b2[:nnz].long()
    ch1, ch2 = torch.bucketize(x, off, right=True), torch.bucketize(y, off, right=True)
    m = {"INTRA": ch1 == ch2, "GW": torch.ones_like(x, dtype=torch.bool), "INTER": ch1 != ch2}[scope]
    stored = 2 * int(m.sum()) - int((m & (x == y)).sum())
    return stored, int(off[-1])


def cpu_kr_100kb(b1, b2, ct):
    """independent scipy bnewt (the restatement tests/test_gpu_norm.py checks the GPU against) on every chromosome's 100 kb matrix"""
    from test_gpu_norm import bnewt, chrom_parts, sym
    t0 = time.perf_counter()
    ok = 0
    for o, nb, x, y, c in chrom_parts(HG38_LEN, 100000, b1, b2, ct):
        if c.sum() == 0:
            continue
        A = sym(nb, x, y, c)
        kept = np.asarray(A.sum(axis=1)).ravel() > 0
        ok += bnewt(A[kept][:, kept]) is not None
    return (time.perf_counter() - t0) * 1e3, ok


def cpu_gw_kr_100kb(b1, b2, ct):
    """the same bnewt on the 100 kb genome-wide matrix"""
    from test_gpu_norm import bnewt, sym
    nb = sum(l // 100000 + 1 for l in HG38_LEN)
    t0 = time.perf_counter()
    A = sym(nb, b1.astype(np.int64), b2.astype(np.int64), ct.astype(np.float64))
    kept = np.asarray(A.sum(axis=1)).ravel() > 0
    ok = bnewt(A[kept][:, kept]) is not None
    return (time.perf_counter() - t0) * 1e3, ok


def timed(torch, nm, call, bytes_full):
    """one warmed-up call with the kernel timers on -> the record of one type"""
    call()
    nm.enable_timing(True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    status, st = call()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    kt = nm.kernel_times()
    nm.enable_timing(False)
    full_ms, full_n = kt["product"]
    kr_ms, kr_n = kt["kr_product"]
    t = {"total_ms": wall, "products": full_n + kr_n, "build_ms": kt["build"][0],
         "ms_per_full_product": full_ms / full_n, "gbs_full_product": bytes_full / (full_ms / full_n) / 1e6}
    if kr_n:
        kv_ms, _ = kt["kr_vector"]
        kw_ms, steps = kt["kr_wall"]
        t.update({"kr_steps": steps, "kr_outer_max": st.kr_outer_max, "kr_failed": st.kr_failed, "kr_residual_max": st.kr_residual_max,
                  "ms_per_kr_product": kr_ms / kr_n, "kr_vector_kernels_ms": kv_ms, "kr_vector_ms_per_step": kv_ms / steps,
                  "kr_loop_wall_ms": kw_ms, "kr_host_round_trip_share": (kw_ms - kr_ms - kv_ms) / kw_ms if kw_ms else 0.0})
    return t, status


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--pairs", default="20000000,250000000")      # the larger one: >= 10^8 nonzeros at 5 kb
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    import torch
    import microcket_b200 as mk
    mk.lib().require_gpu()
    from bench import measured_peak                                 # the peak bench.py's roofline uses, and its source
    peak, peak_src = measured_peak()
    rec = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "hbm_peak_gbs": peak, "peak_source": peak_src, "sizes": []}
    cpu_ref = None
    for n in [int(s) for s in a.pairs.split(",")]:
        pairs = synth_pairs(torch, n, a.seed)
        b1 = torch.empty(n + 1, dtype=torch.int32, device="cuda"); b2 = torch.empty_like(b1); ct = torch.empty_like(b1)
        ws = mk.PairsWorkspace(n + 1)
        size = {"pairs": n, "resolutions": []}
        for res in DEFAULT_RES:
            nnz = ws.bin(pairs.data_ptr(), n, HG38_LEN, res, b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), n + 1)
            stored, rows = matrix_shape(torch, b1, b2, nnz, res)
            bytes_full = 8 * stored + 16 * rows
            row = {"res": res, "nnz": nnz, "stored_entries": stored, "rows": rows, "bytes_per_full_product": bytes_full, "types": {}}
            nm = mk.Norm(HG38_LEN, res, nnz)
            out = torch.empty(rows, dtype=torch.float64, device="cuda")
            for typ in ("VC", "VC_SQRT", "KR"):
                kw = {"d_" + typ.lower(): out.data_ptr()}
                t, status = timed(torch, nm, lambda: nm.run(b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), nnz, (typ,), **kw), bytes_full)
                t["share_of_hbm_peak"] = t["gbs_full_product"] / peak
                if typ == "KR":
                    t["failed_chromosomes"] = [i for i, s in enumerate(status) if s == 2]
                row["types"][typ] = t
                print(json.dumps({"pairs": n, "res": res, "type": typ, **{k: v for k, v in t.items() if k != "failed_chromosomes"}}), flush=True)
            for scope in ("GW", "INTER"):
                sstored, _ = matrix_shape(torch, b1, b2, nnz, res, scope)
                sbytes = 8 * sstored + 16 * rows
                row[scope] = {"stored_entries": sstored, "bytes_per_product": sbytes, "types": {}}
                for typ in ("VC", "KR"):
                    kw = {"d_" + typ.lower(): out.data_ptr()}
                    t, status = timed(torch, nm, lambda: nm.run_genome(b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), nnz, scope, (typ,), **kw), sbytes)
                    t["share_of_hbm_peak"] = t["gbs_full_product"] / peak
                    t["status"] = status
                    if typ == "KR" and t.get("kr_steps"):
                        t["gbs_kr_product"] = sbytes / t["ms_per_kr_product"] / 1e6
                        t["kr_vector_over_product"] = t["kr_vector_ms_per_step"] / t["ms_per_kr_product"]
                    row[scope]["types"][typ] = t
                    print(json.dumps({"pairs": n, "res": res, "type": f"{scope}_{typ}", **t}), flush=True)
            nm.close()
            if res == 100000 and n == max(int(s) for s in a.pairs.split(",")):
                host = [x[:nnz].cpu().numpy().astype(np.uint32) for x in (b1, b2, ct)]
                ms, ok = cpu_kr_100kb(*host)
                gms, gok = cpu_gw_kr_100kb(*host)
                cpu_ref = {"pairs": n, "res": 100000, "scipy_bnewt_ms": ms, "chromosomes_balanced": ok,
                           "gpu_kr_total_ms": row["types"]["KR"]["total_ms"],
                           "scipy_gw_bnewt_ms": gms, "gw_balanced": gok, "gpu_gw_kr_total_ms": row["GW"]["types"]["KR"]["total_ms"],
                           "cpu": os.cpu_count()}
                print(json.dumps(cpu_ref), flush=True)
            size["resolutions"].append(row)
        rec["sizes"].append(size)
        ws.close()
        del pairs, b1, b2, ct
        torch.cuda.empty_cache()
    rec["cpu_reference"] = cpu_ref
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
