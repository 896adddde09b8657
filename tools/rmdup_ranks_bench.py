"""Multi-rank SAM-space krmdup (mk_s2p_rmdup_*) beside the single-GPU cfg.rmdup run, on shards resident in HBM.

  python tools/rmdup_ranks_bench.py --out <record.json> [--groups 5000000] [--world N] [--mode flash] [--reps 3]

Shard r = read groups [r G, (r + 1) G) of seeded synthetic SAM (mk_synth_device, 160 duplicates per 1024 groups drawn from
the whole stream, so that duplicates cross shards), followed by the next shard's first group for pass 2.  One rank per GPU;
with fewer GPUs than --world the ranks share them (the record says how many GPUs there were).  One host thread drives every
rank: pass 1 on all, send on all, decide on all, receive on all, pass 2 on all.  Per rank, CUDA events on the rank's stream
around pass 1, around send + decide + receive and around pass 2, scaled to 10^8 read groups; beside them the single-GPU
cfg.rmdup run (one context, mk_s2p_run_device) over rank 0's shard.  Best of --reps after one warm-up.  The card's name and
power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import microcket_b200 as mk  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 and q.stdout.strip() else ["unknown"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--groups", type=int, default=5000000, help="read groups per rank")
    ap.add_argument("--world", type=int, default=0, help="ranks (default: the GPUs, at least 2)")
    ap.add_argument("--mode", default="flash")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch
    ndev = torch.cuda.device_count()
    if ndev == 0:
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    world = a.world or max(ndev, 2)
    G, per = a.groups, 1e8 / a.groups
    opts = mk.synth_opts(dup_per_1024=160, dup_universe=G * world)
    devs = [r % ndev for r in range(world)]
    bufs, body_len, full_len = [], [], []
    for r in range(world):
        with torch.cuda.device(devs[r]):
            extra = 1 if r + 1 < world else 0
            b, n_full = mk.synth_device(torch, 91, a.mode, "hg38", r * G, G + extra, device=devs[r], opts=opts)
            _, n_body = mk.synth_device(torch, 91, a.mode, "hg38", r * G, G, device=devs[r], opts=opts) if extra else (None, n_full)
            bufs.append(b); body_len.append(n_body); full_len.append(n_full)
    torch.cuda.synchronize()
    cap = G + 1024
    xs = [mk.Xchg(world, r, 2 * cap, device=devs[r]) for r in range(world)]
    mk.Xchg.connect_local(xs)
    cfg = lambda d: mk.S2PConfig(mode=a.mode, threads=8, write_sam=False, device=d, sharded=True, rmdup=True, rmdup_capacity=cap)
    ctxs = [mk.Sam2Pairs(cfg(devs[r])) for r in range(world)]
    streams = [torch.cuda.Stream(device=devs[r]) for r in range(world)]
    texts = [torch.empty(full_len[r] + 4096, dtype=torch.uint8, device=f"cuda:{devs[r]}") for r in range(world)]

    def ev(r):
        e = torch.cuda.Event(enable_timing=True)
        e.record(streams[r])
        return e

    best = None
    dup = None
    for rep in range(a.reps + 1):
        for s in ctxs:
            s.reset()
        t = [[None] * 6 for _ in range(world)]
        for r, s in enumerate(ctxs):
            t[r][0] = ev(r)
            s.rmdup_keys_device(bufs[r].data_ptr(), body_len[r], True, stream=streams[r].cuda_stream)
            t[r][1] = ev(r)
        for r, s in enumerate(ctxs):
            t[r][2] = ev(r)
            s.rmdup_send(xs[r], stream=streams[r].cuda_stream)
        for r, s in enumerate(ctxs):
            s.rmdup_decide(xs[r], stream=streams[r].cuda_stream)
        for r, s in enumerate(ctxs):
            s.rmdup_receive(xs[r], stream=streams[r].cuda_stream)
            t[r][3] = ev(r)
        n_pairs = 0
        for r, s in enumerate(ctxs):
            t[r][4] = ev(r)
            io = s.run_device(bufs[r].data_ptr(), full_len[r], True, texts[r].data_ptr(), texts[r].numel(), stream=streams[r].cuda_stream)
            t[r][5] = ev(r)
            n_pairs += io.n_pairs
        torch.cuda.synchronize()
        ms = [[t[r][0].elapsed_time(t[r][1]), t[r][2].elapsed_time(t[r][3]), t[r][4].elapsed_time(t[r][5])] for r in range(world)]
        dd = [s.rmdup_stats() for s in ctxs]
        dup = (sum(d.uniq for d in dd), sum(d.dup for d in dd), sum(d.discard for d in dd), n_pairs)
        if rep and (best is None or sum(map(sum, ms)) < sum(map(sum, best))):
            best = ms
    for s in ctxs:
        s.close()
    for x in xs:
        x.close()
    # the single-GPU cfg.rmdup run over rank 0's shard (its own key table: per lane)
    with torch.cuda.device(devs[0]):
        one = mk.Sam2Pairs(mk.S2PConfig(mode=a.mode, threads=8, write_sam=False, device=devs[0], rmdup=True, rmdup_capacity=cap))
        st0 = torch.cuda.Stream(device=devs[0])
        one_ms = None
        for rep in range(a.reps + 1):
            one.reset()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(st0)
            one.run_device(bufs[0].data_ptr(), full_len[0], True, texts[0].data_ptr(), texts[0].numel(), stream=st0.cuda_stream)
            e1.record(st0)
            torch.cuda.synchronize()
            if rep and (one_ms is None or e0.elapsed_time(e1) < one_ms):
                one_ms = e0.elapsed_time(e1)
        one.close()
    rec = {
        "tool": "tools/rmdup_ranks_bench.py", "card": card(), "gpus": ndev, "world": world,
        "ranks_share_gpus": world > ndev, "mode": a.mode, "groups_per_rank": G,
        "shard_bytes": body_len, "krmdup_sum": {"uniq": dup[0], "dup": dup[1], "discard": dup[2]}, "pairs_emitted": dup[3],
        "ms_per_1e8_groups_per_rank": [{"rank": r, "device": devs[r], "pass1": best[r][0] * per, "send_decide_receive": best[r][1] * per,
                                        "pass2": best[r][2] * per} for r in range(world)],
        "single_gpu_rmdup_ms_per_1e8_groups": one_ms * per,
        "note": "device time from CUDA events on each rank's stream; best of %d after one warm-up. send + decide + receive on a rank "
                "includes its wait for the other ranks, which one host thread drives in rank order." % a.reps,
    }
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
