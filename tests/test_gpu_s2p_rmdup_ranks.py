"""Multi-rank SAM-space krmdup (mk_s2p_rmdup_*): shards of whole read groups on several ranks (here all in ONE process on one
GPU, joined by mk_xchg_connect_local), one first-occurrence decision over the whole stream.  The ranks' text and SAM
passthrough, concatenated in rank order, must be those of ONE cfg.rmdup context over the whole stream and of the replay
krmdup -> filter -> sam2pairs; their logs must add up to the single run's logs."""
import os
import random
import sys

import pytest

import microcket_b200 as mk
from test_gpu_s2p_rmdup import expected, gpu, same

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import sam_rmdup_oracle as R  # noqa: E402
from rmdup_cases import crafted  # noqa: E402

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

LOG_FIELDS = ("lowMap", "manyHits", "unpaired", "selfCircle", "trans", "cis10K", "cis1K", "cis0")


def _passes_filter(line, min_mapq=10):
    f = line.split(b"\t")
    return len(f) > 5 and f[1].isdigit() and f[4].isdigit() and int(f[4]) >= min_mapq and not (int(f[1]) & 0x700)


def shards_at(sam, run_cuts):
    """Cut `sam` before the QNAME runs `run_cuts` (non-decreasing; equal cuts give empty shards).  → [(body, appended)]: every
    shard but the last is followed by the next shards' lines up to and including their first run with a kept record (the
    read group that lets the shard's own last group be processed)."""
    rs, lines = R.runs(sam)
    starts = [0] + [rs[c][0] if c < len(rs) else len(lines) for c in run_cuts] + [len(lines)]
    join = lambda a, b: b"".join(ln + b"\n" for ln in lines[a:b])
    out = []
    for r in range(len(starts) - 1):
        body, app = join(starts[r], starts[r + 1]), b""
        if r + 2 < len(starts):
            k = next((i for i, (a, n, hdr) in enumerate(rs) if a >= starts[r + 1]), len(rs))
            while k < len(rs):
                a, n, hdr = rs[k]
                if not hdr and any(_passes_filter(ln) for ln in lines[a:a + n]):
                    break
                k += 1
            end = rs[k][0] + rs[k][1] if k < len(rs) else len(lines)
            app = join(starts[r + 1], end)
        out.append((body, app))
    assert b"".join(b for b, _ in out) == sam
    return out


def even_cuts(sam, world):
    n = len(R.runs(sam)[0])
    return [n * r // world for r in range(1, world)]


def dev(data):
    t = torch.zeros(len(data) + 64, dtype=torch.uint8, device="cuda")
    if data:
        t[:len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    return t


def run_ranks(sam, mode, cuts, window=0, key=(5, 16, 5, 16), threads=8, cap=1 << 20, xcap=None, p1_calls=1, reverse=False):
    """→ (text, sam passthrough, summed sam2pairs stats as a dict, summed (uniq, dup, discard, pairs), per-rank texts)"""
    shards = shards_at(sam, cuts)
    world = len(shards)
    xs = [mk.Xchg(world, r, xcap or cap) for r in range(world)]
    mk.Xchg.connect_local(xs)
    cfg = dict(mode=mode, threads=threads, write_sam=True, window_bytes=window, sharded=True, rmdup=True, rmdup_capacity=cap, key=key)
    ctxs = [mk.Sam2Pairs(mk.S2PConfig(**cfg)) for _ in range(world)]
    try:
        for s, (body, _) in zip(ctxs, shards):                 # pass 1, in p1_calls calls that continue where the last stopped
            off = 0
            for c in range(p1_calls, 0, -1):
                rest = body[off:]
                n = len(rest) if c == 1 else rest.rfind(b"\n", 0, len(rest) // c) + 1
                off += s.rmdup_keys_device(dev(rest[:n]).data_ptr(), n, c == 1)
                if c == 1:
                    assert off == len(body)
        for s, x in zip(ctxs, xs):
            s.rmdup_send(x)
        order = range(world - 1, -1, -1) if reverse else range(world)
        for r in order:
            ctxs[r].rmdup_decide(xs[r])
        for s, x in zip(ctxs, xs):
            s.rmdup_receive(x)
        texts, sams = [], []
        for s, (body, app) in zip(ctxs, shards):               # pass 2 over the shard and its boundary group
            data = body + app
            d = dev(data)
            text = torch.empty(len(data) + 4096, dtype=torch.uint8, device="cuda")
            so = torch.empty(len(data) + 64, dtype=torch.uint8, device="cuda")
            io = s.run_device(d.data_ptr(), len(data), True, text.data_ptr(), text.numel(), 0, 0, so.data_ptr(), so.numel())
            texts.append(bytes(text[:io.pairs_text_len].cpu().numpy().tobytes()))
            sams.append(bytes(so[:io.sam_text_len].cpu().numpy().tobytes()))
        counts = [s.finish(0, 0).groups for s in ctxs]
        total, base = sum(counts), 0
        st = {f: 0 for f in LOG_FIELDS + ("groups",)}
        for s, c in zip(ctxs, counts):
            x = s.finish(base, total)
            base += c
            for f in st:
                st[f] += getattr(x, f)
        dd = [s.rmdup_stats() for s in ctxs]
        dsum = tuple(sum(getattr(d, f) for d in dd) for f in ("uniq", "dup", "discard", "pairs"))
        return b"".join(texts), b"".join(sams), st, dsum, texts
    finally:
        for s in ctxs:
            s.close()
        for x in xs:
            x.close()


def check(got, exp):
    p, so, st, dsum, _ = got
    ep, eso, est, edd = exp
    assert dsum[:3] == (edd.uniq, edd.dup, edd.discard) and dsum[3] == sum(dsum[:3])
    for f in LOG_FIELDS + ("groups",):
        assert st[f] == getattr(est, f), f
    assert p == ep
    assert so == eso


@pytest.mark.parametrize("mode,genome,seed", [("flash", "hg38", 51), ("unc", "hg38", 52), ("unc", "mm10", 53), ("flash", "mm10", 54)])
def test_world_sizes_equal_one_context_and_the_replay(oracle, mode, genome, seed):
    n = 24000
    sam = mk.synth_host(seed, mode, genome, 0, n, mk.synth_opts(dup_per_1024=160, dup_universe=n))
    e = expected(oracle, sam, mode)
    one = gpu(sam, mode)
    same(one, e)
    outs = []
    for world in (1, 2, 3, 8):
        got = run_ranks(sam, mode, even_cuts(sam, world))
        check(got, e)
        outs.append(got[:4])
        if world > 1:                                          # per lane (one krmdup per shard) would have removed fewer
            lane_dup = 0
            for body, _ in shards_at(sam, even_cuts(sam, world)):
                lane_dup += oracle.krmdup(R.sam_to_fastq(body)[0])[2].dup
            assert got[3][1] > lane_dup
    assert all(o == outs[0] for o in outs)


@pytest.mark.parametrize("mode", ["unc", "flash"])
def test_small_windows_and_pass1_in_several_calls(oracle, mode):
    n = 12000
    sam = mk.synth_host(61, mode, "hg38", 0, n, mk.synth_opts(dup_per_1024=200, dup_universe=n))
    e = expected(oracle, sam, mode)
    for window, calls in ((1 << 20, 2), (1 << 16, 3)):
        check(run_ranks(sam, mode, even_cuts(sam, 3), window=window, p1_calls=calls), e)


def _fq_read(rng, n):
    return bytes(rng.choice(b"ACGT") for _ in range(n))


def _pair(q, r1, r2, pos, mode):
    """one read pair's SAM lines (mapq 60, forward strand)"""
    if mode == "flash":
        return b"\t".join([q, b"0", b"chr1", b"%d" % pos, b"60", b"%dM" % len(r1), b"*", b"0", b"0", r1, b"F" * len(r1)]) + b"\n"
    return (b"\t".join([q, b"65", b"chr1", b"%d" % pos, b"60", b"%dM" % len(r1), b"=", b"1", b"0", r1, b"F" * len(r1)]) + b"\n" +
            b"\t".join([q, b"129", b"chr1", b"%d" % (pos + 300), b"60", b"%dM" % len(r2), b"=", b"1", b"0", r2, b"F" * len(r2)]) + b"\n")


@pytest.mark.parametrize("mode", ["unc", "flash"])
def test_crafted_keys_across_ranks(oracle, mode):
    """Cross-rank first occurrences: copies on ranks 1 and 2 of a pair first seen on rank 0, two copies inside rank 1 of a pair
    also on rank 0, the lower-case (tag) identity space on different ranks, the all-G pair (all-ones 64-bit key with
    key=(0,16,0,16)), a rank whose shard is only discards and an empty shard."""
    rng = random.Random(99 + len(mode))
    key = (0, 16, 0, 16)
    fill = lambda k: [(_fq_read(rng, 60), _fq_read(rng, 60)) for _ in range(k)]
    a, b, g = (_fq_read(rng, 60), _fq_read(rng, 60)), (_fq_read(rng, 60), _fq_read(rng, 60)), (b"G" * 60, b"G" * 60)
    low = (b"a" + a[0][1:], a[1])                               # a's bases, lower-case first base: another identity space
    disc = [(_fq_read(rng, 10), _fq_read(rng, 60)) for _ in range(30)]        # short mate 1: discarded
    ranks = [[a, b, g, low] + fill(40),                          # rank 0: first occurrences
             fill(20) + [a, b, b] + fill(20) + [a, g],            # rank 1: copies of rank-0 pairs, two of b inside the rank
             fill(10) + [a, low, low, g] + fill(10),              # rank 2: more copies, the tag space's copies
             [],                                                  # rank 3: empty
             disc,                                                # rank 4: only discards
             fill(30) + [low, b, g]]                              # rank 5
    if mode == "flash":
        ranks = [[(r1, R.revcomp(r1)) for r1, _ in rk] for rk in ranks]
    lines, cuts, k = [b"@HD\tVN:1.6\n", b"@SQ\tSN:chr1\tLN:248956422\n"], [], 2
    for r, rk in enumerate(ranks):
        if r:
            cuts.append(k)
        for r1, r2 in rk:
            lines.append(_pair(b"q%d" % k, r1, r2, rng.randrange(1000, 200000000), mode))
            k += 1
    sam = b"".join(lines)
    e = expected(oracle, sam, mode, key=key)
    assert e[3].dup >= 12 and e[3].discard >= 30
    same(gpu(sam, mode, key=key), e)
    for reverse in (False, True):
        check(run_ranks(sam, mode, cuts, key=key, reverse=reverse), e)
    # the generic crafted corpus (N, lower case, short mates, missing mates, supplementary records) on 3 ranks
    sam2, _ = crafted(random.Random(7 + len(mode)), 3000, mode)
    e2 = expected(oracle, sam2, mode, threads=4)
    check(run_ranks(sam2, mode, even_cuts(sam2, 3), threads=4, window=1 << 16), e2)


def test_refusals():
    n = 3000
    sam = mk.synth_host(71, "unc", "hg38", 0, n, mk.synth_opts(dup_per_1024=160, dup_universe=n))
    shards = shards_at(sam, even_cuts(sam, 2))
    cfg = lambda cap: mk.S2PConfig(mode="unc", threads=8, write_sam=False, sharded=True, rmdup=True, rmdup_capacity=cap)

    def ranks(cap=1 << 16, xcap=1 << 16):
        xs = [mk.Xchg(2, r, xcap) for r in range(2)]
        mk.Xchg.connect_local(xs)
        return [mk.Sam2Pairs(cfg(cap)) for _ in range(2)], xs

    def close(ctxs, xs):
        for o in ctxs + xs:
            o.close()

    bufs = [dev(b) for b, _ in shards]
    text = torch.empty(len(sam) + 4096, dtype=torch.uint8, device="cuda")
    # steps out of order, and a context without cfg.rmdup
    ctxs, xs = ranks()
    with pytest.raises(mk.MkError, match="error -5"):
        ctxs[0].rmdup_send(xs[0])
    plain = mk.Sam2Pairs(mk.S2PConfig(mode="unc", threads=8))
    with pytest.raises(mk.MkError, match="error -5"):
        plain.rmdup_keys_device(bufs[0].data_ptr(), len(shards[0][0]), True)
    plain.close()
    for s, (b, _), d in zip(ctxs, shards, bufs):
        s.rmdup_keys_device(d.data_ptr(), len(b), True)
    with pytest.raises(mk.MkError, match="error -5"):               # pass 2 before receive
        ctxs[0].run_device(bufs[0].data_ptr(), len(shards[0][0]), True, text.data_ptr(), text.numel())
    with pytest.raises(mk.MkError, match="error -5"):
        ctxs[0].push(b"", True)
    with pytest.raises(mk.MkError, match="error -5"):
        ctxs[0].rmdup_decide(xs[0])
    for s, x in zip(ctxs, xs):
        s.rmdup_send(x)
    for s, x in zip(ctxs, xs):
        s.rmdup_decide(x)
    for s, x in zip(ctxs, xs):
        s.rmdup_receive(x)
    # pass-2 bytes whose lines differ from pass 1's: rank 1's shard given to rank 0
    with pytest.raises(mk.MkError, match="error -6"):
        ctxs[0].run_device(bufs[1].data_ptr(), len(shards[1][0]), True, text.data_ptr(), text.numel())
    close(ctxs, xs)
    # more read pairs in a shard than cfg.rmdup_capacity
    ctxs, xs = ranks(cap=100)
    with pytest.raises(mk.MkError, match="error -4"):
        ctxs[0].rmdup_keys_device(bufs[0].data_ptr(), len(shards[0][0]), True)
    close(ctxs, xs)
    # an owner sent more key records than its exchange capacity
    ctxs, xs = ranks(xcap=64)
    for s, (b, _), d in zip(ctxs, shards, bufs):
        s.rmdup_keys_device(d.data_ptr(), len(b), True)
    for s, x in zip(ctxs, xs):
        s.rmdup_send(x)
    for s, x in zip(ctxs, xs):
        with pytest.raises(mk.MkError, match="error -4"):
            s.rmdup_decide(x)
    close(ctxs, xs)
