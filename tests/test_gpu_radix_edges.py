"""The radix sort (csrc/radix_sort.cuh) directly, and every consumer of it through the C ABI, at the inputs where a sort goes wrong.

Random pairs make every byte pass run and never land near a tile edge.  The sort's data-dependent paths are elsewhere: a pass whose
digit is the same for every key is skipped by the device plan, which changes the buffer the next pass reads, the buffer that
holds the result (final_buf) and the pass that writes the index values (iota_vals); with no pass at all (n_exec == 0) the values
are never written.  Padding items of the last tile take digit 255 and must rank after real keys with digit 255.

The sort itself is reached through tests/radix_harness.cu, built into a temporary directory; the reference is a numpy stable
lexsort over the scheduled bytes, least significant pass first, and every comparison is exact.  The consumers are compared with
the C oracle (tests/oracle_lib.py), the numpy restatements of tests/test_gpu_pairs.py and ref_norms of tests/test_gpu_norm.py."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import microcket_b200 as mk

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "microcket_b200", "csrc")
HARNESS = os.path.join(ROOT, "tests", "radix_harness.cu")
TILE = {"kv64": 256 * 16, "rec16": 256 * 8}                 # RS_THREADS * ITEMS of the two policies
UQ_TILE = 256 * 8                                             # k_uniq_cells / k_unique_rec16 / k_rle_heads tiles (pairs.cu)
SENT32 = 0xA5A5A5A5


# ---------------------------------------------------------------- the harness
@pytest.fixture(scope="module")
def harness_so(tmp_path_factory):
    """<tmp>/libradix_harness.so, linked against the library only for its error plumbing and SM count"""
    mk.build()
    d = tmp_path_factory.mktemp("radix_harness")
    lib_dir = os.path.dirname(mk.LIB_PATH)
    so = str(d / "libradix_harness.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared",
           "-I", CSRC, HARNESS, "-L" + lib_dir, "-lmicrocket_b200", "-Xlinker", "-rpath=" + lib_dir, "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return so


def test_harness_compiles(harness_so):
    """radix_sort.cuh and mk_common.cuh still build for sm_100a outside the library (no GPU needed)"""
    assert os.path.getsize(harness_so) > 0


class Radix:
    def __init__(self, so):
        mk.lib().require_gpu()
        L = self.L = C.CDLL(so)
        vp, P = C.c_void_p, C.POINTER
        L.rh_last_error.restype = C.c_char_p
        L.rh_sort_kv64.argtypes = [vp, vp, vp, vp, C.c_uint64, P(C.c_int), C.c_int, C.c_int, C.c_size_t, P(C.c_uint32), P(C.c_uint64)]
        L.rh_sort_rec16.argtypes = [vp, vp, C.c_uint64, P(C.c_int), C.c_int, C.c_int, C.c_size_t, P(C.c_uint32), P(C.c_uint64)]

    def kv64(self, k0, k1, v0, v1, n, sched, iota, ws_n):
        out, launches = (C.c_uint32 * 2)(), C.c_uint64()
        rc = self.L.rh_sort_kv64(k0, k1, v0, v1, n, (C.c_int * len(sched))(*sched), len(sched), iota, ws_n, out, C.byref(launches))
        return rc, out[0], out[1], launches.value

    def rec16(self, k0, k1, n, sched, hist_done, ws_n):
        out, launches = (C.c_uint32 * 2)(), C.c_uint64()
        rc = self.L.rh_sort_rec16(k0, k1, n, (C.c_int * len(sched))(*sched), len(sched), int(hist_done), ws_n, out, C.byref(launches))
        return rc, out[0], out[1], launches.value

    def error(self):
        return self.L.rh_last_error().decode()


@pytest.fixture(scope="module")
def radix(harness_so):
    return Radix(harness_so)


# ---------------------------------------------------------------- host predictions
def ref_perm(kb, sched):
    """stable LSD order of the rows of kb (n x key bytes, uint8) on the scheduled bytes: np.lexsort's last key is the primary one"""
    if len(kb) == 0:
        return np.zeros(0, dtype=np.int64)
    return np.lexsort([kb[:, b] for b in sched])


def predict_plan(kb, sched):
    """(n_exec, final_buf) as k_radix_plan decides them: a pass runs unless every key has the same digit there"""
    if len(kb) == 0:
        return 0, 0
    n_exec = sum(int((kb[:, b] != kb[0, b]).any()) for b in sched)
    return n_exec, n_exec & 1


def make_keys(structure, n, nbytes, sched, seed):
    """n rows of nbytes key bytes (uint8); the structure is laid on the scheduled bytes, the others stay random (carried along)"""
    rng = np.random.default_rng(seed)
    kb = rng.integers(0, 256, (n, nbytes), dtype=np.uint8)
    s = list(sched)
    if n == 0 or structure == "random":
        return kb
    if structure == "equal":
        kb[:, s] = kb[0, s]
    elif structure in ("const_first", "const_mid", "const_last"):
        p = {"const_first": 0, "const_mid": len(s) // 2, "const_last": len(s) - 1}[structure]
        kb[:, s[p]] = 0x5C
    elif structure == "two":                                  # two keys only: runs of equal keys cross many tiles
        pick = rng.random(n) < 0.5
        kb[:, s] = np.where(pick[:, None], kb[0, s], kb[1, s])
    elif structure in ("sorted", "reverse"):
        kb = kb[ref_perm(kb, s)]
        if structure == "reverse":
            kb = kb[::-1].copy()
    elif structure == "pad255":                               # digit 255 everywhere; one pass runs, mostly 255 there too
        kb[:, s] = 255
        p = len(s) // 2
        other = rng.random(n) < 0.125
        kb[other, s[p]] = rng.integers(0, 255, int(other.sum()), dtype=np.uint8)
        kb[-1, s[p]] = 255
        kb[0, s[p]] = 3
    elif structure == "one_off":                              # every key in one digit bucket but one key
        kb[:, s] = 7
        kb[n // 2, s[len(s) // 2]] = 200
    else:
        raise ValueError(structure)
    return kb


def expected_n_exec(structure, n, sched):
    """what each structure is built to make the plan do (asserted against the host prediction, so a case cannot drift)"""
    if n == 0 or structure == "equal":
        return 0
    if structure in ("pad255", "one_off"):
        return 1 if n > 1 else 0
    if structure.startswith("const_"):
        return len(sched) - 1
    return None


# ---------------------------------------------------------------- running the harness
def dev_u8(a, extra=0):
    b = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    t = torch.full((len(b) + extra,), 0x5A, dtype=torch.uint8, device="cuda")
    if len(b):
        t[:len(b)] = torch.from_numpy(b.copy()).cuda()
    return t


def host_u8(t, nbytes):
    return t[:nbytes].cpu().numpy()


def run_kv64(radix, kb, sched, iota, ws_n=None):
    n = len(kb)
    keys = np.ascontiguousarray(kb).view(np.uint64).reshape(-1)
    vals = np.random.default_rng(n).integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32)
    k0 = dev_u8(keys, 64); k1 = dev_u8(np.zeros(0, np.uint8), max(n, 8) * 8 + 64)
    v0 = dev_u8(vals, 64) if not iota else dev_u8(np.full(n, SENT32, np.uint32), 64)
    v1 = dev_u8(np.zeros(0, np.uint8), max(n, 8) * 4 + 64)
    before = [t.clone() for t in (k0, k1, v0, v1)]
    rc, fb, ne, launches = radix.kv64(k0.data_ptr(), k1.data_ptr(), v0.data_ptr(), v1.data_ptr(), n, sched, iota, ws_n or max(n, 1))
    assert rc == 0, radix.error()
    perm = ref_perm(kb, sched)
    assert (ne, fb) == predict_plan(kb, sched)
    assert launches == 2 + (len(sched) if n else 0)           # histogram + plan, then one (possibly empty) kernel per pass
    if n == 0:                                                # nothing to sort: no pass ran and no buffer was written
        for a, b in zip(before, (k0, k1, v0, v1)):
            assert torch.equal(a, b)
        return ne, fb
    ko = (k1 if fb else k0); vo = (v1 if fb else v0)
    got_k = host_u8(ko, n * 8).view(np.uint64)
    got_v = host_u8(vo, n * 4).view(np.uint32)
    assert np.array_equal(got_k, keys[perm])
    if not iota:
        assert np.array_equal(got_v, vals[perm])              # values travel with their keys
    elif ne:
        assert np.array_equal(got_v, perm.astype(np.uint32))  # the stable permutation, written by the first executed pass
    else:
        # the contract when no pass runs: the permutation is the identity and the values are NOT written (v[0] keeps what the
        # caller left there); a consumer reads the index itself (pairs.cu k_mark_first, norm.cu k_nm_fill_lower)
        assert np.array_equal(got_v, np.full(n, SENT32, np.uint32))
    # the other buffer's tail beyond n is never written
    for t, w in ((k0, 8), (k1, 8), (v0, 4), (v1, 4)):
        assert (t[n * w:].cpu().numpy() == 0x5A).all()
    return ne, fb


def run_rec16(radix, kb, sched, hist_done, ws_n=None):
    n = len(kb)
    k0 = dev_u8(kb, 64); k1 = dev_u8(np.zeros(0, np.uint8), max(n, 8) * 16 + 64)
    before = [k0.clone(), k1.clone()]
    rc, fb, ne, launches = radix.rec16(k0.data_ptr(), k1.data_ptr(), n, sched, hist_done, ws_n or max(n, 1))
    assert rc == 0, radix.error()
    assert (ne, fb) == predict_plan(kb, sched)
    assert launches == (0 if hist_done else 1) + 1 + (len(sched) if n else 0)
    if n == 0:
        assert torch.equal(before[0], k0) and torch.equal(before[1], k1)
        return ne, fb
    got = host_u8(k1 if fb else k0, n * 16).reshape(n, 16)
    assert np.array_equal(got, kb[ref_perm(kb, sched)])          # whole records: the unscheduled bytes are carried along
    for t in (k0, k1):
        assert (t[n * 16:].cpu().numpy() == 0x5A).all()
    return ne, fb


# ---------------------------------------------------------------- the sort: sizes
SIZES = [0, 1, 31, 32, 33, 2047, 2048, 2049, 4095, 4096, 4097, 3 * 2048 + 17, 3 * 4096 + 17, (1 << 20) + 7]
KV_SCHED = list(range(8))
REC_SCHED = list(range(9))                                    # 69-bit keys of the dedup + binning sort


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("policy", ["kv64", "rec16", "rec16_hist"])
def test_sort_sizes(radix, policy, n):
    kb = make_keys("random", n, 8 if policy == "kv64" else 16, KV_SCHED if policy == "kv64" else REC_SCHED, seed=n)
    if policy == "kv64":
        kb[:, 6:] &= 0x03                                    # a few equal high bytes (duplicates at small n come from below)
        if n > 64:
            kb[n // 3: n // 3 + 40] = kb[n // 3]             # a run of equal keys: stability
        run_kv64(radix, kb, KV_SCHED, iota=1)
    else:
        if n > 64:
            kb[n // 3: n // 3 + 40, :9] = kb[n // 3, :9]
        run_rec16(radix, kb, REC_SCHED, hist_done=policy == "rec16_hist")


# ---------------------------------------------------------------- the sort: key structure
STRUCTURES = ["equal", "const_first", "const_mid", "const_last", "two", "sorted", "reverse", "pad255", "one_off"]


@pytest.mark.gpu
@pytest.mark.parametrize("structure", STRUCTURES)
@pytest.mark.parametrize("policy", ["kv64_iota", "kv64_vals", "kv64_3bytes", "rec16", "rec16_hist"])
def test_sort_key_structure(radix, policy, structure):
    kv = policy.startswith("kv64")
    tile = TILE["kv64" if kv else "rec16"]
    n = 5 * tile + 17 if structure != "two" else (1 << 18) + 3          # last tile partly padding; "two": runs over ~64 tiles
    sched = [0, 1, 2] if policy == "kv64_3bytes" else (KV_SCHED if kv else REC_SCHED)
    kb = make_keys(structure, n, 8 if kv else 16, sched, seed=len(structure))
    exp = expected_n_exec(structure, n, sched)
    pred, _ = predict_plan(kb, sched)
    if exp is not None:
        assert pred == exp, (structure, pred)
    if kv:
        ne, _ = run_kv64(radix, kb, sched, iota=0 if policy == "kv64_vals" else 1)
    else:
        ne, _ = run_rec16(radix, kb, sched, hist_done=policy == "rec16_hist")
    assert ne == pred


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 4096, 4097])
def test_sort_all_equal_values_contract(radix, n):
    """n_exec == 0 with iota_vals: keys stay in buffer 0 and the value buffers are not written at all"""
    kb = make_keys("equal", n, 8, KV_SCHED, seed=3)
    assert run_kv64(radix, kb, KV_SCHED, iota=1) == (0, 0)


# ---------------------------------------------------------------- the sort: schedules
SCHEDULES = {
    "contiguous69": list(range(9)),
    "noncontiguous": [3, 0, 9, 14, 6],
    "bytes8to15": list(range(8, 16)),
    "no_top_word": list(range(12)),                           # the index word (bytes 12..15) is carried, as in k_pack_keys
}


@pytest.mark.gpu
@pytest.mark.parametrize("structure", ["random", "const_mid", "two"])
@pytest.mark.parametrize("hist_done", [False, True])
@pytest.mark.parametrize("name", list(SCHEDULES))
def test_sort_schedules(radix, name, hist_done, structure):
    sched = SCHEDULES[name]
    n = 3 * TILE["rec16"] + 17
    kb = make_keys(structure, n, 16, sched, seed=11)
    if name == "no_top_word":
        kb[:, 12:] = np.arange(n, dtype=np.uint32).view(np.uint8).reshape(n, 4)
    if structure == "random":
        kb[:, sched] &= 0x0F                                  # small digits: many ties broken by input order
    ne, _ = run_rec16(radix, kb, sched, hist_done)
    if structure == "const_mid":
        assert ne == len(sched) - 1


@pytest.mark.gpu
def test_sort_kv64_noncontiguous_and_top_byte(radix):
    n = 3 * TILE["kv64"] + 17
    kb = make_keys("random", n, 8, [7, 2, 5], seed=5)
    kb[:, [7, 2, 5]] &= 0x07
    run_kv64(radix, kb, [7, 2, 5], iota=1)
    run_kv64(radix, kb, [7, 2, 5], iota=0)


@pytest.mark.gpu
def test_sort_refusals(radix):
    """n >= 2^30 and n > the workspace are refused before anything is launched (the workspace here holds 1000 elements)"""
    buf = torch.zeros(1024, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr()
    for n, ws_n, what in (((1 << 30), 1000, "2^30"), ((1 << 30) + 5, 1000, "2^30"), (1001, 1000, "workspace")):
        rc, _, _, launches = radix.kv64(p, p, p, p, n, KV_SCHED, 1, ws_n)
        assert rc == -4 and launches == 0 and what in radix.error()
        for hist_done in (False, True):
            rc, _, _, launches = radix.rec16(p, p, n, REC_SCHED, hist_done, ws_n)
            assert rc == -4 and launches == 0 and what in radix.error()
    assert (buf.cpu().numpy() == 0).all()


@pytest.mark.gpu
def test_sort_bench_size_rec16(radix):
    """~1e8 16-byte records on 69 key bits, histograms taken by the caller: the size and key width of the benchmark's sort.
    With the input index in the unsorted top word, "sorted on (key, index) and a permutation of the input" is exactly the
    stable sort, so it is checked on the device."""
    n = 97_800_000
    g = torch.Generator(device="cuda"); g.manual_seed(12)
    keys = torch.empty((n // 4, 3), dtype=torch.int32, device="cuda")     # n / 4 distinct keys: every key ~4 times, scattered
    keys[:, :2] = torch.randint(-2**31, 2**31, (n // 4, 2), dtype=torch.int32, device="cuda", generator=g)
    keys[:, 2] = torch.randint(0, 32, (n // 4,), dtype=torch.int32, device="cuda", generator=g)
    rec = torch.empty((n, 4), dtype=torch.int32, device="cuda")
    rec[:, :3] = keys[torch.randint(0, n // 4, (n,), device="cuda", generator=g)]
    rec[:, 3] = torch.arange(n, dtype=torch.int32, device="cuda")
    del keys
    src = rec.clone()
    alt = torch.empty_like(rec)
    rc, fb, ne, _ = radix.rec16(rec.data_ptr(), alt.data_ptr(), n, REC_SCHED, True, n)
    assert rc == 0, radix.error()
    assert ne == 9 and fb == 1
    out = alt if fb else rec
    u = lambda c: out[:, c].to(torch.int64) & 0xFFFFFFFF
    z, y, x, w = u(2), u(1), u(0), u(3)
    lt = w[:-1] < w[1:]
    for col in (x, y, z):
        lt = (col[:-1] < col[1:]) | ((col[:-1] == col[1:]) & lt)
    assert bool(lt.all())                                     # strictly increasing in (key, input index): sorted and stable
    seen = torch.zeros(n, dtype=torch.bool, device="cuda")
    seen[w] = True
    assert bool(seen.all())                                   # n distinct indices: a permutation
    assert torch.equal(out, src[w])                           # every record is its input record


# ================================================================ consumers, through the C ABI
from oracle_lib import Pair  # noqa: E402
from test_gpu_pairs import HG38_LEN  # noqa: E402

TOY_LEN = [3000000]                                           # 31 bins at 100 kb: 5 + 5 + 17 + 17 + 3 = 47 key bits, 6 passes


def pairs_of(rows):
    """(chr1, pos1, chr2, pos2, strands, lane) rows -> mk_pair records, cls by the rule unpack_key applies"""
    p = np.zeros(len(rows), dtype=mk.PAIR_DTYPE)
    if len(rows):
        a = np.array(rows, dtype=np.int64)
        p["chr1"], p["pos1"], p["chr2"], p["pos2"], p["strands"], p["lane"] = a.T
    d = (p["pos2"].astype(np.int64) - p["pos1"].astype(np.int64)) & 0xFFFFFFFF
    p["cls"] = np.where(p["chr1"] != p["chr2"], 0, np.where(d >= 10000, 1, np.where(d >= 1000, 2, 3)))
    return p


def to_dev(p, extra=16):
    return dev_u8(p, extra)


def as_oracle(p):
    return (Pair * max(len(p), 1)).from_buffer_copy(p.tobytes() if len(p) else bytes(16))


def bits_for(v):
    b = 1
    while b < 64 and (v >> b):
        b += 1
    return b


def packed_key_bytes(p, lens, res, max_lane=0):
    """numpy / Python restatement of k_pack_keys (PackCfg, put_bits) for keyable pairs -> (key bytes n x 12, scheduled passes)"""
    off = np.concatenate([[0], np.cumsum(np.array(lens, dtype=np.int64) // res + 1)])
    nb, nr, nl = bits_for(int(off[-1])), bits_for(res - 1), (bits_for(max_lane) if max_lane else 0)
    total = 2 * nb + 2 * nr + nl + 3
    rows = []
    for r in p:
        a, b = int(off[r["chr1"]] + r["pos1"] // res), int(off[r["chr2"]] + r["pos2"] // res)
        r1, r2, st, sw = int(r["pos1"] % res), int(r["pos2"] % res), int(r["strands"]) & 3, 0
        if a > b:
            a, b, r1, r2, st, sw = b, a, r2, r1, ((st & 1) << 1) | (st >> 1), 1
        k = a
        for v, w in ((b, nb), (int(r["lane"]), nl), (r1, nr), (r2, nr), (sw, 1), (st, 2)):
            k = (k << w) | v
        rows.append(list(k.to_bytes(12, "little")))
    return np.array(rows, dtype=np.uint8).reshape(-1, 12), (total + 7) // 8


def dedup_bin_case(oracle, p, lens, res, max_lane=0, bad=None, cap=None, expect_error=False):
    """mk_pairs_dedup_bin_indexed_device on p against the oracle: keep, kept_idx, the decoded kept pairs and the COO, exactly.
    bad: the pairs that cannot be keyed (left out of the oracle's input, counted by mk_pairs_dropped)"""
    n = len(p)
    ok = np.ones(n, dtype=bool) if bad is None else ~bad
    good = p[ok]
    keep, kept = oracle.coord_dedup(as_oracle(good), len(good))
    exp_keep = np.zeros(n, dtype=np.uint8)
    exp_keep[ok] = np.frombuffer(bytes(keep), dtype=np.uint8)[:len(good)]
    b1, b2, ct = oracle.bin_coo(as_oracle(good), len(good), keep, lens, res) if len(good) else ([], [], [])
    cap = len(b1) if cap is None else cap
    ws = mk.PairsWorkspace(n)
    d = to_dev(p)
    o = [torch.full((n + 8,), -1, dtype=torch.int32, device="cuda") for _ in range(3)]
    d_keep = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    d_idx = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    args = (d.data_ptr(), n, lens, res, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), cap)
    kw = dict(max_lane=max_lane, d_keep=d_keep.data_ptr(), d_kept_idx=d_idx.data_ptr())
    try:
        if expect_error:
            with pytest.raises(mk.MkError, match="error -4"):
                ws.dedup_bin(*args, **kw)
            for t in o:
                assert (t[cap:].cpu().numpy() == -1).all()   # nothing written past the capacity
            return
        got, nnz = ws.dedup_bin(*args, **kw)
        assert (got, nnz, ws.dropped()) == (kept, len(b1), n - len(good))
        assert np.array_equal(d_keep.cpu().numpy(), exp_keep)
        idx = d_idx[:got].cpu().numpy().astype(np.uint32)
        out = np.frombuffer(d[:got * 16].cpu().numpy().tobytes(), dtype=mk.PAIR_DTYPE)
        assert np.array_equal(out, p[idx])                    # every kept pair is, field for field, the input pair kept_idx names
        assert np.array_equal(np.sort(idx), np.flatnonzero(exp_keep))
        for t, e in zip(o, (b1, b2, ct)):
            assert t[:nnz].cpu().numpy().astype(np.uint32).tolist() == list(e)
            assert (t[cap:].cpu().numpy() == -1).all()
    finally:
        ws.close()


# ---------------------------------------------------------------- mk_pairs_dedup_bin_indexed_device
def variant_pairs(genome, variant, n, seed):
    """one (bin1, bin2) cell; 'identical': one pair n times (no pass runs); 'strands': only the strands differ (byte 0: one
    pass); 'strands_pos2': strands and pos2 % res in bits 5 and up (bytes 0 and 1: two passes)"""
    rng = np.random.default_rng(seed)
    c, pos1, pos2 = (0, 1_000_000, 1_000_003) if genome == "hg38" else (0, 250_000, 250_003)
    st = np.full(n, 1) if variant == "identical" else rng.integers(0, 4, n)
    p2 = pos2 + (32 * rng.integers(0, 3, n) if variant == "strands_pos2" else np.zeros(n, dtype=np.int64))
    return pairs_of([(c, pos1, c, int(q), int(s), 0) for q, s in zip(p2, st)])


@pytest.mark.gpu
@pytest.mark.parametrize("variant,n_exec", [("identical", 0), ("strands", 1), ("strands_pos2", 2)])
@pytest.mark.parametrize("genome", ["hg38", "toy"])
def test_dedup_bin_pass_parity(oracle, genome, variant, n_exec):
    """all four combinations of n_pass odd / even (keys packed in place or not) and executed passes odd / even (the result in
    the pairs buffer or the workspace: both branches of k_copy_if_alt), on runs and one cell longer than several k_uniq_cells tiles"""
    lens, res = (HG38_LEN, 5000) if genome == "hg38" else (TOY_LEN, 100000)
    n = 3 * UQ_TILE + 17
    p = variant_pairs(genome, variant, n, seed=n_exec)
    kb, n_pass = packed_key_bytes(p, lens, res)
    assert n_pass == (9 if genome == "hg38" else 6)
    assert predict_plan(kb, range(n_pass))[0] == n_exec
    dedup_bin_case(oracle, p, lens, res)


@pytest.mark.gpu
def test_dedup_bin_coordinate_edges(oracle):
    """pos 0 and pos == chromosome length (the last bin) on both sides, inter- and intra-chromosomal, duplicated"""
    rng = np.random.default_rng(4)
    L = HG38_LEN
    rows = []
    for _ in range(3000):
        c1, c2 = sorted(rng.integers(0, 25, 2).tolist())
        e1 = [0, L[c1], int(rng.integers(0, L[c1] + 1))][rng.integers(0, 3)]
        e2 = [0, L[c2], int(rng.integers(0, L[c2] + 1))][rng.integers(0, 3)]
        if c1 == c2 and e1 > e2:
            e1, e2 = e2, e1
        rows.append((c1, e1, c2, e2, int(rng.integers(0, 4)), 0))
    rows += rows[:500]
    p = pairs_of(rows)
    assert ((p["pos2"] == np.array(L)[p["chr2"]]) & (p["pos1"] == 0)).any()
    dedup_bin_case(oracle, p, L, 5000)


@pytest.mark.gpu
def test_dedup_bin_res_1_and_equal_lanes(oracle):
    """res = 1 (pos % res has one bit, always 0); max_lane > 0 while every pair has the same lane (the lane field is constant)"""
    rng = np.random.default_rng(6)
    lens = [3000000, 5000]
    rows = [(c, int(a), c, int(a) + int(d), int(s), 0) for c, a, d, s in
            zip(rng.integers(0, 2, 5000), rng.integers(0, 4000, 5000), rng.integers(0, 600, 5000), rng.integers(0, 4, 5000))]
    p = pairs_of(rows + rows[:1000])
    dedup_bin_case(oracle, p, lens, 1)
    q = p.copy(); q["lane"] = 2
    dedup_bin_case(oracle, q, lens, 1, max_lane=3)


@pytest.mark.gpu
def test_dedup_bin_unkeyable(oracle):
    """only unkeyable pairs: nothing kept, no cell, all counted as dropped, keep all 0; unkeyable pairs plus one cell"""
    n = 3 * UQ_TILE + 5
    rng = np.random.default_rng(8)
    rows = [(25 + int(rng.integers(0, 3)), 100, 0, 200, 0, 0) for _ in range(n)]
    p = pairs_of(rows)
    dedup_bin_case(oracle, p, HG38_LEN, 5000, bad=np.ones(n, dtype=bool))
    cell = [(2, 1_000_000 + i % 7, 2, 1_000_500, i % 4, 0) for i in range(300)]
    order = rng.permutation(n + 300)
    p = pairs_of(rows + cell)[order]
    bad = (np.arange(n + 300) < n)[order]
    dedup_bin_case(oracle, p, HG38_LEN, 5000, bad=bad)


@pytest.mark.gpu
def test_dedup_bin_capacity(oracle):
    from test_gpu_pairs import random_pairs
    p = random_pairs(20000, 31, dup_frac=0.3)
    keep, _ = oracle.coord_dedup(as_oracle(p), len(p))
    nnz = len(oracle.bin_coo(as_oracle(p), len(p), keep, HG38_LEN, 5000)[0])
    dedup_bin_case(oracle, p, HG38_LEN, 5000, cap=nnz)                       # exactly enough: accepted
    dedup_bin_case(oracle, p, HG38_LEN, 5000, cap=nnz - 1, expect_error=True)


# ---------------------------------------------------------------- mk_pairs_dedup_device
DEDUP_SCHED = [12, 4, 5, 6, 7, 10, 11, 0, 1, 2, 3, 8, 9, 14, 15]      # pairs.cu: strands, pos2, chr2, pos1, chr1, lane


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2047, 2048, 2049])
@pytest.mark.parametrize("variant,n_exec", [("identical", 0), ("lane", 1), ("strands_lane", 2)])
def test_pairs_dedup_skipped_passes(oracle, variant, n_exec, n):
    """no pass (the result reaches d_pairs through the host's final_buf == 0 copy), one pass (the run heads are written straight
    into d_pairs) and two passes (final_buf == 0 again, after passes)"""
    rng = np.random.default_rng(n)
    lane = rng.integers(0, 3, n) if variant != "identical" else np.zeros(n, dtype=np.int64)
    st = rng.integers(0, 4, n) if variant == "strands_lane" else np.full(n, 2)
    p = pairs_of([(4, 77_000, 9, 5_000, int(s), int(l)) for s, l in zip(st, lane)])
    assert predict_plan(np.ascontiguousarray(p).view(np.uint8).reshape(n, 16), DEDUP_SCHED)[0] == n_exec
    keep, kept = oracle.coord_dedup(as_oracle(p), n)
    ws = mk.PairsWorkspace(n)
    d = to_dev(p)
    got = ws.dedup(d.data_ptr(), n)
    ws.close()
    assert got == kept
    out = np.frombuffer(d[:got * 16].cpu().numpy().tobytes(), dtype=mk.PAIR_DTYPE)
    exp = p[np.frombuffer(bytes(keep), dtype=np.uint8)[:n] == 1]
    order = np.lexsort((exp["strands"], exp["pos2"], exp["chr2"], exp["pos1"], exp["chr1"], exp["lane"]))
    assert np.array_equal(out, exp[order])


# ---------------------------------------------------------------- mk_pairs_bin_device
def bin_case(oracle, p, lens, res, bad=None, cap=None, expect_error=False):
    n = len(p)
    ok = np.ones(n, dtype=bool) if bad is None else ~bad
    good = p[ok]
    b1, b2, ct = oracle.bin_coo(as_oracle(good), len(good), None, lens, res) if len(good) else ([], [], [])
    cap = len(b1) if cap is None else cap
    ws = mk.PairsWorkspace(n)
    d = to_dev(p)
    o = [torch.full((n + 8,), -1, dtype=torch.int32, device="cuda") for _ in range(3)]
    args = (d.data_ptr(), n, lens, res, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), cap)
    try:
        if expect_error:
            with pytest.raises(mk.MkError, match="error -4"):
                ws.bin(*args)
        else:
            nnz = ws.bin(*args)
            assert nnz == len(b1) and ws.dropped() == n - len(good)
            for t, e in zip(o, (b1, b2, ct)):
                assert t[:nnz].cpu().numpy().astype(np.uint32).tolist() == list(e)
        for t in o:
            assert (t[cap:].cpu().numpy() == -1).all()
    finally:
        ws.close()
    return b1, ct


@pytest.mark.gpu
def test_bin_one_cell_and_long_runs(oracle):
    n = 3 * UQ_TILE + 5
    rng = np.random.default_rng(2)
    one = pairs_of([(3, 5_000_000 + int(a), 3, 5_004_000 + int(b), 0, 0) for a, b in zip(rng.integers(0, 5000, n), rng.integers(0, 1000, n))])
    off = np.concatenate([[0], np.cumsum(np.array(HG38_LEN) // 5000 + 1)])
    keys = (off[one["chr1"]] + one["pos1"] // 5000).astype(np.uint64) << np.uint64(32) | (off[one["chr2"]] + one["pos2"] // 5000).astype(np.uint64)
    assert predict_plan(keys.view(np.uint8).reshape(n, 8), [0, 1, 2, 4, 5, 6])[0] == 0       # every pass skipped
    b1, ct = bin_case(oracle, one, HG38_LEN, 5000)
    assert ct == [n]
    cells = [(1, 0, 1, 7), (1, 7, 1, 5000), (6, 100, 20, 3)]
    pick = rng.integers(0, 3, 3 * 2500)
    p = pairs_of([(cells[k][0], cells[k][1], cells[k][2], cells[k][3], 0, 0) for k in pick])
    _, ct = bin_case(oracle, p, HG38_LEN, 5000)
    assert sorted(ct) == sorted(np.bincount(pick).tolist())


@pytest.mark.gpu
def test_bin_sentinel_only_and_capacity(oracle):
    n = UQ_TILE + 3
    p = pairs_of([(30, 5, 0, 5, 0, 0)] * n)
    b1, _ = bin_case(oracle, p, HG38_LEN, 5000, bad=np.ones(n, dtype=bool))
    assert b1 == []
    from test_gpu_pairs import random_pairs
    q = random_pairs(30000, 17)
    nnz = len(oracle.bin_coo(as_oracle(q), len(q), None, HG38_LEN, 100000)[0])
    bin_case(oracle, q, HG38_LEN, 100000, cap=nnz)
    bin_case(oracle, q, HG38_LEN, 100000, cap=nnz - 1, expect_error=True)


# ---------------------------------------------------------------- mk_dedup_keys_device
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 4095, 4096, 4097, 3 * 4096 + 17])
@pytest.mark.parametrize("structure", ["random", "one_byte", "top_byte"])
def test_key_dedup_edges(structure, n):
    rng = np.random.default_rng(n)
    kb = rng.integers(0, 256, (n, 8), dtype=np.uint8)
    if structure != "random":
        kb[:] = kb[0]
        b = 3 if structure == "one_byte" else 7
        kb[:, b] = rng.integers(0, 5, n)                      # one byte varies: one pass, many duplicates
        assert predict_plan(kb, range(8))[0] == (1 if len(np.unique(kb[:, b])) > 1 else 0)
    keys = kb.view(np.uint64).reshape(-1)
    keys[rng.integers(0, n, n // 3)] = keys[rng.integers(0, n, n // 3)]
    _, first = np.unique(keys, return_index=True)
    exp = np.zeros(n, dtype=np.uint8); exp[first] = 1
    L = mk.lib()
    d = torch.from_numpy(keys.view(np.int64).copy()).cuda()
    keep = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    nu = C.c_uint64()
    L.check(L.L.mk_dedup_keys_device(0, d.data_ptr(), n, keep.data_ptr(), C.byref(nu), None))
    assert nu.value == len(first) and np.array_equal(keep.cpu().numpy(), exp)


# ---------------------------------------------------------------- mk_norm_device
NORM_TYPES = ("VC", "VC_SQRT", "KR")


def mirror_keys(lens, res, b1, b2):
    """the keys k_nm_classify gives norm.cu's sort: bin2 for a mirrored entry (intra-chromosomal, off the diagonal), nb otherwise"""
    off = np.concatenate([[0], np.cumsum(np.array(lens, dtype=np.int64) // res + 1)])
    nb = int(off[-1])
    c1 = np.searchsorted(off, b1, side="right") - 1
    c2 = np.searchsorted(off, b2, side="right") - 1
    keys = np.where((c1 == c2) & (b1 != b2), b2, nb).astype(np.uint64)
    n_pass = (nb.bit_length() + 7) // 8
    return keys, n_pass


def norm_run(nm, coo, pad_to=0):
    """one mk_norm_device call on a device COO whose arrays are zero-padded to pad_to entries -> ({type: vector}, status)"""
    m = len(coo[0])
    d = [torch.zeros(max(m, pad_to, 1), dtype=torch.int32, device="cuda") for _ in range(3)]
    for t, a in zip(d, coo):
        if m:
            t[:m] = torch.from_numpy(np.asarray(a, dtype=np.uint32).view(np.int32).copy()).cuda()
    outs = {t: torch.full((nm.n_bins,), -1.0, dtype=torch.float64, device="cuda") for t in NORM_TYPES}
    status, _ = nm.run(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), m, NORM_TYPES,
                       **{("d_" + t.lower()): outs[t].data_ptr() for t in NORM_TYPES})
    return {t: v.cpu().numpy() for t, v in outs.items()}, status


def assert_norms(lens, res, coo, got, status, rtol_vc=1e-12):
    from test_gpu_norm import ref_norms
    exp, est = ref_norms(lens, res, *(np.asarray(a, dtype=np.int64) for a in coo))
    assert status == est
    for t in ("VC", "VC_SQRT"):
        np.testing.assert_allclose(got[t], exp[t], rtol=rtol_vc, atol=0, err_msg=t)
    assert np.array_equal(np.isnan(got["KR"]), np.isnan(exp["KR"]))
    np.testing.assert_allclose(got["KR"], exp["KR"], rtol=1e-5)


NORM_LENS, NORM_RES = [40_000_000], 100_000                  # 401 bins: the sort's keys take two bytes


def first_coo(seed=1):
    """a COO whose mirrored entries make both passes of norm.cu's sort run, so that d_vals[0] ends up holding a permutation;
    rows 0..4 hold only their diagonal, so every mirrored entry's COO index is >= 5"""
    rng = np.random.default_rng(seed)
    nb = 401
    i = rng.integers(5, nb, 6000); j = rng.integers(5, nb, 6000)
    cells = set(zip(np.minimum(i, j).tolist(), np.maximum(i, j).tolist())) | {(k, k) for k in range(nb)}
    cells = sorted(cells)
    b1 = np.array([c[0] for c in cells]); b2 = np.array([c[1] for c in cells])
    return b1, b2, rng.integers(1, 60, len(cells))


def star_coos():
    """every entry intra-chromosomal, off the diagonal and in one column bin2: every key equal, no pass runs (n_exec == 0)"""
    return [(np.array([0, 1, 2]), np.array([5, 5, 5]), np.array([3, 11, 40])), (np.array([0]), np.array([3]), np.array([7]))]


@pytest.mark.gpu
def test_norm_reused_object_when_no_sort_pass_runs():
    """A reused mk_norm whose sort runs no pass must not build the mirrored half from the previous call's permutation.  The
    second call's device arrays are zero-padded to the first call's length, so stale indices stay in bounds and show up as
    wrong vectors."""
    b1, b2, ct = first_coo()
    keys, n_pass = mirror_keys(NORM_LENS, NORM_RES, b1, b2)
    kb = keys.view(np.uint8).reshape(-1, 8)
    assert predict_plan(kb, range(n_pass)) == (2, 0)          # d_vals[0] holds the first call's permutation afterwards
    stale = ref_perm(kb, range(n_pass))
    assert stale[0] >= 5                                      # what an unguarded read of d_vals[0] would take as entry indices
    nm = mk.Norm(NORM_LENS, NORM_RES, len(b1))
    try:
        got, status = norm_run(nm, (b1, b2, ct))
        assert_norms(NORM_LENS, NORM_RES, (b1, b2, ct), got, status)
        for coo in star_coos():
            k2, _ = mirror_keys(NORM_LENS, NORM_RES, coo[0], coo[1])
            assert predict_plan(k2.view(np.uint8).reshape(-1, 8), range(n_pass))[0] == 0
            got, status = norm_run(nm, coo, pad_to=len(b1))
            assert_norms(NORM_LENS, NORM_RES, coo, got, status)
            fresh = mk.Norm(NORM_LENS, NORM_RES, len(b1))
            again, status2 = norm_run(fresh, coo)
            fresh.close()
            assert status2 == status
            for t in NORM_TYPES:
                assert got[t].tobytes() == again[t].tobytes(), t
    finally:
        nm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", [0, 1])
def test_norm_fresh_object_when_no_sort_pass_runs(which):
    coo = star_coos()[which]
    nm = mk.Norm(NORM_LENS, NORM_RES, 8)
    try:
        got, status = norm_run(nm, coo)
    finally:
        nm.close()
    assert_norms(NORM_LENS, NORM_RES, coo, got, status)
    if which == 1:                                            # a single entry (0, 3): KR balances it, VC is its count
        assert status == [0] and got["VC"][0] > 0 and np.isfinite(got["KR"][[0, 3]]).all()


@pytest.mark.gpu
def test_norm_csr_edges():
    """Rows of exactly 96, 97, 128 and 129 stored entries (the four-loads-in-flight loop of k_nm_spmv starts at k + 96 < end),
    in the upper half (row 0) and in the mirrored half (the last row) of their chromosome; a chromosome boundary exactly at the
    4096-bin tile edge of k_nm_row_ptr; a one-bin chromosome holding only its diagonal; a few inter-chromosomal entries.
    Integer counts make every row sum exact, so VC and VC_SQRT are held to 1e-13 whatever the order of summation."""
    res = 1000
    row_lens = [96, 97, 128, 129]
    lens = [4095 * res] + [(L - 1) * res for L in row_lens] + [500]
    off = np.concatenate([[0], np.cumsum(np.array(lens, dtype=np.int64) // res + 1)])
    assert off[1] == 4096 and list(np.diff(off)[1:]) == row_lens + [1]
    rng = np.random.default_rng(3)
    cells = set()
    i = rng.integers(0, 4096, 30000); j = np.minimum(i + rng.integers(0, 300, 30000), 4095)
    cells |= set(zip(i.tolist(), j.tolist())) | {(k, k) for k in range(4096)} | {(4094, 4095)}
    for c, L in enumerate(row_lens, start=1):
        o = int(off[c])
        cells |= {(o, o + k) for k in range(L)}                   # row 0: L upper entries
        cells |= {(o + k, o + L - 1) for k in range(1, L)}         # last row: L - 1 mirrored entries and its diagonal
        cells |= {(o + k, o + k) for k in range(1, L - 1)}
    one = int(off[5])
    cells |= {(one, one)}
    cells |= {(10, 4096), (4095, 4096), (4096 + 5, one), (0, one)}            # inter-chromosomal: not part of any matrix
    cells = sorted(cells)
    b1 = np.array([c[0] for c in cells]); b2 = np.array([c[1] for c in cells]); ct = rng.integers(1, 1000, len(cells))
    intra = np.searchsorted(off, b1, side="right") == np.searchsorted(off, b2, side="right")
    # stored entries per CSR row, both halves
    lengths = np.bincount(np.concatenate([b1[intra & (b1 != b2)], b2[intra]]), minlength=int(off[-1]))
    for c, L in enumerate(row_lens, start=1):
        assert lengths[off[c]] == L and lengths[off[c + 1] - 1] == L
    nm = mk.Norm(lens, res, len(b1))
    try:
        got, status = norm_run(nm, (b1, b2, ct))
    finally:
        nm.close()
    assert status == [0] * 6
    assert_norms(lens, res, (b1, b2, ct), got, status, rtol_vc=1e-13)


# ---------------------------------------------------------------- krmdup (dedup.cu)
@pytest.mark.gpu
@pytest.mark.parametrize("n", [2047, 2048, 2049, 3 * 2048 + 17])
@pytest.mark.parametrize("variant", ["identical", "two"])
def test_krmdup_equal_keys(oracle, variant, n):
    """every read pair the same (no sort pass runs: k_fq_mark reads buffer 0 as sorted), or one of two read pairs (runs of
    equal keys across the sort's tiles), at Rec16 tile edges: read1, read2 and the log equal the oracle's"""
    recs = mk.synth_host(5, "fastq", "hg38", 0, 2).split(b"\n@")
    pair_a = recs[0] + b"\n@" + recs[1] + b"\n"
    pair_b = b"@" + recs[2] + b"\n@" + recs[3].rstrip(b"\n") + b"\n"
    pick = np.random.default_rng(n).random(n) < 0.5 if variant == "two" else np.zeros(n, dtype=bool)
    fq = b"".join(pair_b if q else pair_a for q in pick)
    o1, o2, ost = oracle.krmdup(fq)
    k = mk.Krmdup()
    try:
        r1, r2, st = k.run(fq)
    finally:
        k.close()
    assert r1 == o1 and r2 == o2 and st.log_text() == ost.log_text()
    assert st.uniq == (2 if variant == "two" else 1)
