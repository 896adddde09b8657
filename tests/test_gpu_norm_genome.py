"""Genome-wide balancing (csrc/norm.cu through capi.Norm.run_genome and `pairs2bins -n`): GW_VC / GW_KR over the whole-genome
matrix and INTER_VC / INTER_KR over its inter-chromosomal entries, against an independent numpy / scipy restatement (the
`bnewt`, `sym` and `sum_factor` of test_gpu_norm) on COO made by the library's own binning of seeded pairs.  PARITY UNPINNED."""
import os
import re
import subprocess

import numpy as np
import pytest

import microcket_b200 as mk
from hic_norm_check import check_norm
from test_gpu_norm import BIN, NAMES, TYPES, bnewt, gpu_coo, gpu_norms, host, sum_factor, sym, toy_pairs
from test_gpu_pairs import HG38_LEN, random_pairs

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SCOPES = ("GW", "INTER")
SLICE = 2048                      # NM_GS in norm.cu: rows per slice of the genome-wide segment


# ---------------------------------------------------------------- independent restatement
def scope_matrix(lens, res, b1, b2, ct, scope):
    """-> (n_bins, upper-triangle entries x, y, c of the scope's matrix in global bins)"""
    off = np.concatenate([[0], np.cumsum(np.array(lens, dtype=np.int64) // res + 1)])
    b1, b2, ct = (np.asarray(a, dtype=np.int64) for a in (b1, b2, ct))
    m = np.ones(len(b1), dtype=bool)
    if scope == "INTER":
        m = np.searchsorted(off, b1, side="right") != np.searchsorted(off, b2, side="right")
    return int(off[-1]), b1[m], b2[m], ct[m].astype(np.float64)


def ref_genome(lens, res, b1, b2, ct, scope):
    """-> ({"VC", "KR": vector over all bins}, status) by the restatement"""
    nb, x, y, c = scope_matrix(lens, res, b1, b2, ct, scope)
    if c.sum() == 0:
        return {"VC": np.zeros(nb), "KR": np.full(nb, np.nan)}, 1
    A = sym(nb, x, y, c)
    rs = np.asarray(A.sum(axis=1)).ravel()
    out = {"VC": sum_factor(rs.copy(), x, y, c), "KR": np.full(nb, np.nan)}
    kept = rs > 0
    xk = bnewt(A[kept][:, kept])
    if xk is None:
        return out, 2
    n = np.full(nb, np.nan); n[kept] = 1 / xk
    out["KR"] = sum_factor(n, x, y, c)
    return out, 0


def balanced(lens, res, b1, b2, ct, scope, kr):
    """row sums of A / (n n^T) constant on kept rows; the normalised matrix sums to the raw one"""
    nb, x, y, c = scope_matrix(lens, res, b1, b2, ct, scope)
    A = sym(nb, x, y, c)
    kept = np.isfinite(kr)
    assert np.array_equal(kept, np.asarray(A.sum(axis=1)).ravel() > 0)
    inv = np.where(kept, 1 / np.where(kept, kr, 1), 0)
    rows = inv * (A @ inv)
    assert np.ptp(rows[kept]) <= 1e-5 * rows[kept].mean(), np.ptp(rows[kept]) / rows[kept].mean()
    w = np.where(x != y, 2.0, 1.0)
    assert np.isclose((c * w / (kr[x] * kr[y])).sum(), (c * w).sum(), rtol=1e-9)


# ---------------------------------------------------------------- GPU side
def gpu_genome(lens, res, b1, b2, ct, nnz, scope, types=("VC", "KR"), nm=None):
    own = nm is None
    if own:
        nm = mk.Norm(lens, res, max(nnz, 1))
    outs = {t: torch.full((nm.n_bins,), -1.0, dtype=torch.float64, device="cuda") for t in types}
    status, st = nm.run_genome(b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), nnz, scope, types,
                               **{("d_" + t.lower()): outs[t].data_ptr() for t in types})
    if own:
        nm.close()
    return {t: v.cpu().numpy() for t, v in outs.items()}, status, st


def check_against_ref(lens, res, b1, b2, ct, nnz, scope, want_status=0):
    got, status, st = gpu_genome(lens, res, b1, b2, ct, nnz, scope)
    hb = [host(a, nnz) for a in (b1, b2, ct)]
    exp, est = ref_genome(lens, res, *hb, scope)
    assert status == est == want_status, (status, est)
    np.testing.assert_allclose(got["VC"], exp["VC"], rtol=1e-12, atol=0)
    assert np.array_equal(np.isnan(got["KR"]), np.isnan(exp["KR"]))
    np.testing.assert_allclose(got["KR"], exp["KR"], rtol=1e-5)
    if status == 0:
        balanced(lens, res, *hb, scope, got["KR"])
        assert st.kr_failed == 0 and st.kr_residual_max <= 1e-6 and st.kr_matvecs > 0
    return got, st


# ---------------------------------------------------------------- tests
@pytest.mark.parametrize("res", [1000000, 100000])
@pytest.mark.parametrize("scope", SCOPES)
def test_hg38(res, scope):
    p = random_pairs(2000000, 41)                                   # dense enough at 100 kb for a doubly-stochastic scaling
    b1, b2, ct, nnz = gpu_coo(p, HG38_LEN, res)
    check_against_ref(HG38_LEN, res, b1, b2, ct, nnz, scope)


def test_toy_genome():
    """a chromosome shorter than one bin, one with trans contacts only, one with no contacts at all"""
    lens = [3000000, 2200000, 40000, 950000, 700000]
    res = 100000
    p = toy_pairs(lens, 60000, 43, skip=(3,))
    p = p[(p["chr1"] != 4) & (p["chr2"] != 4)]
    b1, b2, ct, nnz = gpu_coo(p, lens, res)
    _, intra_status, _ = gpu_norms(lens, res, b1, b2, ct, nnz)
    assert intra_status == [0, 0, 0, 1, 1]
    off = np.cumsum([0] + [l // res + 1 for l in lens])
    for scope in SCOPES:
        got, _ = check_against_ref(lens, res, b1, b2, ct, nnz, scope)
        for t in ("VC", "KR"):
            assert (got[t][off[3]:off[4]] > 0).all()                 # trans only: GW / INTER vectors all the same
            assert not (got[t][off[4]:off[5]] > 0).any()             # no contacts: no valid norm


def test_one_chromosome_and_no_trans():
    """no inter entries: INTER has no matrix; GW of one chromosome is its intra vectors, of several a per-chromosome multiple"""
    res = 100000
    lens = [3000000]
    b1, b2, ct, nnz = gpu_coo(toy_pairs(lens, 40000, 45), lens, res)
    intra, _, _ = gpu_norms(lens, res, b1, b2, ct, nnz, ("VC", "KR"))
    gw, status, _ = gpu_genome(lens, res, b1, b2, ct, nnz, "GW")
    assert status == 0
    np.testing.assert_allclose(gw["VC"], intra["VC"], rtol=1e-12)
    assert np.array_equal(np.isnan(gw["KR"]), np.isnan(intra["KR"]))
    np.testing.assert_allclose(gw["KR"], intra["KR"], rtol=1e-5)
    inter, status, _ = gpu_genome(lens, res, b1, b2, ct, nnz, "INTER")
    assert status == 1 and (inter["VC"] == 0).all() and np.isnan(inter["KR"]).all()

    lens = [3000000, 2200000, 900000]
    b1, b2, ct, nnz = gpu_coo(toy_pairs(lens, 60000, 46, trans=0.0), lens, res)
    intra, _, _ = gpu_norms(lens, res, b1, b2, ct, nnz, ("VC", "KR"))
    _, status, _ = gpu_genome(lens, res, b1, b2, ct, nnz, "INTER")
    assert status == 1
    gw, _ = check_against_ref(lens, res, b1, b2, ct, nnz, "GW")
    off = np.cumsum([0] + [l // res + 1 for l in lens])
    for t, tol in (("VC", 1e-12), ("KR", 1e-5)):
        for c in range(len(lens)):
            g, i = gw[t][off[c]:off[c + 1]], intra[t][off[c]:off[c + 1]]
            ok = np.isfinite(i) & (i > 0)
            r = g[ok] / i[ok]
            assert np.ptp(r) <= tol * r.mean(), (t, c)               # one sum factor for the genome, one per chromosome


def test_kr_failure():
    """an inter-only path 0 - 1 - 2 across three one-bin chromosomes has no doubly-stochastic scaling"""
    lens = [50000, 50000, 50000]
    res = 100000
    d = [torch.tensor(np.array(a, dtype=np.int32), device="cuda") for a in ([0, 1], [1, 2], [5, 7])]
    got, status, st = gpu_genome(lens, res, *d, 2, "INTER")
    assert status == 2 and st.kr_failed == 1
    assert np.isnan(got["KR"]).all()
    vc = np.array([5.0, 12.0, 7.0])
    np.testing.assert_allclose(got["VC"], sum_factor(vc, np.array([0, 1]), np.array([1, 2]), np.array([5.0, 7.0])), rtol=1e-12)
    _, est = ref_genome(lens, res, [0, 1], [1, 2], [5, 7], "INTER")
    assert est == 2


@pytest.mark.parametrize("extra", [-1, 0, 1, None])
def test_slice_edges(extra):
    """bin counts of 2 slices - 1, 2 slices, 2 slices + 1, and less than one slice; three chromosomes of about a third each (the
    inter-chromosomal matrix of two chromosomes of unequal size has no doubly-stochastic scaling)"""
    res = 1000
    target = 1500 if extra is None else 2 * SLICE + extra
    k = target // 3
    lens = [(k - 1) * res + 500, (k - 1) * res + 500, (target - 2 * k - 1) * res + 500]
    assert sum(l // res + 1 for l in lens) == target
    b1, b2, ct, nnz = gpu_coo(toy_pairs(lens, 200000, 47, trans=0.3), lens, res)
    for scope in SCOPES:
        check_against_ref(lens, res, b1, b2, ct, nnz, scope)


def test_bitwise_reproducible():
    p = random_pairs(2000000, 48)
    res = 100000
    b1, b2, ct, nnz = gpu_coo(p, HG38_LEN, res)
    moved = [torch.empty(nnz + 977, dtype=torch.int32, device="cuda")[977:] for _ in range(3)]
    for m, a in zip(moved, (b1, b2, ct)):
        m.copy_(a[:nnz])
    firsts = {}
    for scope in SCOPES:
        first, s1, _ = gpu_genome(HG38_LEN, res, b1, b2, ct, nnz, scope)
        firsts[scope] = first
        again, s2, _ = gpu_genome(HG38_LEN, res, b1, b2, ct, nnz, scope)
        other, s3, _ = gpu_genome(HG38_LEN, res, *moved, nnz, scope)
        assert s1 == s2 == s3 == 0
        for t in ("VC", "KR"):
            assert first[t].tobytes() == again[t].tobytes() == other[t].tobytes(), (scope, t)
    # a reused object: intra, genome, intra; the intra bits are a fresh object's
    fresh, fs, _ = gpu_norms(HG38_LEN, res, b1, b2, ct, nnz)
    nm = mk.Norm(HG38_LEN, res, nnz)
    outs = {t: torch.empty(nm.n_bins, dtype=torch.float64, device="cuda") for t in TYPES}
    kw = {("d_" + t.lower()): outs[t].data_ptr() for t in TYPES}
    nm.run(b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), nnz, TYPES, **kw)
    g1, _, _ = gpu_genome(HG38_LEN, res, b1, b2, ct, nnz, "GW", nm=nm)
    status, _ = nm.run(b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), nnz, TYPES, **kw)
    g2, _, _ = gpu_genome(HG38_LEN, res, b1, b2, ct, nnz, "GW", nm=nm)
    nm.close()
    assert status == fs
    for t in TYPES:
        assert outs[t].cpu().numpy().tobytes() == fresh[t].tobytes(), t
    for t in ("VC", "KR"):
        assert g1[t].tobytes() == g2[t].tobytes() == firsts["GW"][t].tobytes(), t


def test_hg38_5kb_genome_wide():
    """>= 20 M pairs at 5 kb (the lockstep size): 617 669 rows, one segment over 302 slices"""
    p = random_pairs(20000000, 49, dup_frac=0.0)
    res = 5000
    b1, b2, ct, nnz = gpu_coo(p, HG38_LEN, res)
    got, status, st = gpu_genome(HG38_LEN, res, b1, b2, ct, nnz, "GW")
    assert status == 0 and st.kr_residual_max <= 1e-6 and st.kr_outer_max >= 2
    assert -(-len(got["VC"]) // SLICE) > 148
    hb = [host(a, nnz) for a in (b1, b2, ct)]
    nb, x, y, c = scope_matrix(HG38_LEN, res, *hb, "GW")
    rs = np.asarray(sym(nb, x, y, c).sum(axis=1)).ravel()
    np.testing.assert_allclose(got["VC"], sum_factor(rs, x, y, c), rtol=1e-12)
    balanced(HG38_LEN, res, *hb, "GW", got["KR"])


def test_refusals():
    lens = [1000000, 500000]
    res = 100000                                                    # 11 + 6 bins
    ok = [torch.tensor(np.array(a, dtype=np.int32), device="cuda") for a in ([0, 1, 12], [1, 5, 16], [3, 4, 5])]
    out = [torch.empty(17, dtype=torch.float64, device="cuda") for _ in range(2)]
    nm = mk.Norm(lens, res, 3)
    args = [a.data_ptr() for a in ok] + [3]
    kw = dict(d_vc=out[0].data_ptr(), d_kr=out[1].data_ptr())
    assert nm.run_genome(*args, "GW", ("VC", "KR"), **kw)[0] in (0, 2)
    for scope, types, k in (("GW", ("VC_SQRT",), kw), ("INTER", ("VC", 8), kw), (0, ("VC",), kw), (3, ("VC",), kw),
                            ("GW", ("VC", "KR"), dict(d_vc=out[0].data_ptr())), ("INTER", ("VC",), dict(d_kr=out[1].data_ptr()))):
        with pytest.raises(mk.MkError, match="error -1"):
            nm.run_genome(*args, scope, types, **k)
    for bad in (([0, 1, 12], [1, 5, 17], [3, 4, 5]),                  # a bin past the end
                ([0, 5, 12], [1, 4, 16], [3, 4, 5]),                  # bin1 > bin2
                ([0, 1, 0], [1, 5, 16], [3, 4, 5])):                   # not sorted
        t = [torch.tensor(np.array(a, dtype=np.int32), device="cuda") for a in bad]
        with pytest.raises(mk.MkError, match="error -1"):
            nm.run_genome(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), 3, "GW", ("VC",), **kw)
    nm.close()
    nm = mk.Norm(lens, res, 2)
    with pytest.raises(mk.MkError, match="error -4"):
        nm.run_genome(*args, "INTER", ("VC",), **kw)
    nm.close()


# ---------------------------------------------------------------- pairs2bins -n
def run(cmd, **kw):
    return subprocess.run(cmd, capture_output=True, **kw)


def stored_genome(vals, status, kind, lens, res):
    off = np.cumsum([0] + [l // res + 1 for l in lens])
    ok = status == 0 or (status == 2 and kind == "VC")
    return [ok and bool((np.isfinite(vals[off[c]:off[c + 1]]) & (vals[off[c]:off[c + 1]] > 0)).any()) for c in range(len(lens))]


def test_pairs2bins_all_seven_types(tmp_path):
    """dense (1 Mb, 100 kb), sort path (50 kb) and -d (5 kb) resolutions with the seven types; the file's vectors are byte-equal
    to the library's on the .coo the run wrote, and everything before the normalised section is the file without -n"""
    p = toy_pairs(HG38_LEN, 300000, 51)
    p = p[(p["chr1"] != NAMES.index("chrM")) & (p["chr2"] != NAMES.index("chrM"))]     # one chromosome without contacts
    lines = [f"r{i}\t{NAMES[a]}\t{x}\t{NAMES[b]}\t{y}\t+\t-\n" for i, (a, x, b, y) in enumerate(zip(p["chr1"].tolist(), p["pos1"].tolist(), p["chr2"].tolist(), p["pos2"].tolist()))]
    pf = tmp_path / "x.pairs"; pf.write_text("## pairs format v1.0\n" + "".join(lines + lines[:5000]))
    info = tmp_path / "hg38.info"; info.write_text("".join(f"{n}\t{l}\n" for n, l in zip(NAMES, HG38_LEN)))
    res = [1000000, 100000, 50000, 5000]
    args = ["-r", ",".join(map(str, res)), str(pf)]
    exe = os.path.join(BIN, "pairs2bins")
    r = run([exe, "-d", "-H", str(tmp_path / "n.hic"), "-n", "INTER_KR,VC,GW_VC,VC_SQRT,KR,GW_KR,INTER_VC"] + args + [str(tmp_path / "n"), str(info)])
    assert r.returncode == 0, r.stderr
    err = r.stderr.decode()
    assert err.count("INFO: KR at ") == 4 and "(2 dense)" in err
    for k in ("GW_KR", "INTER_KR"):
        assert err.count(f"INFO: {k} at ") == 4 and all(f"INFO: {k} at {x} bp: " in err for x in res)
        assert re.search(f"INFO: {k} at 1000000 bp: [0-9]+ steps, the matrix balanced\\.", err), err
    r = run([exe, "-d", "-H", str(tmp_path / "p.hic")] + args + [str(tmp_path / "p"), str(info)])
    assert r.returncode == 0, r.stderr
    coo, norms = {}, {}
    for rs in res:
        a = np.loadtxt(tmp_path / f"n.{rs}.coo", dtype=np.int64, ndmin=2)
        coo[rs] = (a[:, 0], a[:, 1], a[:, 2])
        d = [torch.tensor(a[:, k].astype(np.int32), device="cuda") for k in range(3)]
        got, status, _ = gpu_norms(HG38_LEN, rs, *d, len(a))
        norms[rs] = {t: (got[t], [s != 1 if t != "KR" else s == 0 for s in status]) for t in TYPES}
        for scope in SCOPES:
            g, st, _ = gpu_genome(HG38_LEN, rs, *d, len(a), scope)
            for t in ("VC", "KR"):
                norms[rs][f"{scope}_{t}"] = (g[t], stored_genome(g[t], st, t, HG38_LEN, rs))
        m = NAMES.index("chrM")
        assert not any(v[1][m] for v in norms[rs].values())
        assert all(norms[rs][f"{s}_VC"][1][0] for s in SCOPES)
        assert rs != 1000000 or all(norms[rs][f"{s}_KR"][1][0] for s in SCOPES)
    h = check_norm(str(tmp_path / "n.hic"), HG38_LEN, coo, norms)
    assert {k[0] for k in h["vectors"]} == set(TYPES) | {f"{s}_{t}" for s in SCOPES for t in ("VC", "KR")}
    cut = h["section_start"]
    plain = (tmp_path / "p.hic").read_bytes()
    assert (tmp_path / "n.hic").read_bytes()[:cut] == plain[:cut] and plain[cut:] == b"\0" * 8
    for t in ("GW_VC_SQRT", "INTER_VC_SQRT", "GW"):
        assert run([exe, "-H", str(tmp_path / "o.hic"), "-n", t] + args + [str(tmp_path / "o"), str(info)]).returncode == 2


def test_pairs2bins_inter_kr_failure(tmp_path):
    """the inter-only path of test_kr_failure through the CLI: INTER_VC stored, no INTER_KR, and the failure reported"""
    from hic_norm_reader import read_norm
    info = tmp_path / "g.info"; info.write_text("a\t50000\nb\t50000\nc\t50000\n")
    pf = tmp_path / "x.pairs"
    pf.write_text("".join(["r\ta\t10\tb\t10\t+\t-\n"] * 5 + ["r\tb\t10\tc\t10\t+\t-\n"] * 7))
    r = run([os.path.join(BIN, "pairs2bins"), "-H", str(tmp_path / "o.hic"), "-n", "INTER_VC,INTER_KR", "-r", "100000", str(pf), str(tmp_path / "o"), str(info)])
    assert r.returncode == 0, r.stderr
    assert b"INFO: INTER_KR at 100000 bp: " in r.stderr and b"the matrix did not balance." in r.stderr
    vec = read_norm(str(tmp_path / "o.hic"))["vectors"]
    assert sorted(vec) == [("INTER_VC", c, 100000) for c in (1, 2, 3)]
