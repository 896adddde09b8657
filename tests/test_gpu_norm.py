"""Matrix balancing (csrc/norm.cu through capi.Norm and `pairs2bins -n`): VC, VC_SQRT and KR vectors against an independent
numpy / scipy restatement of juicer's published behaviour (Knight & Ruiz `bnewt`, the sum factor), on COO made by the library's
own binning of seeded pairs.  PARITY UNPINNED: juicer_tools is absent, so the restatement is the yardstick."""
import os
import subprocess
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

import microcket_b200 as mk
from hic_norm_check import check_norm
from test_gpu_pairs import HG38_LEN, random_pairs, to_dev

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

BIN = os.path.join(os.path.dirname(mk.LIB_PATH), "bin")
NAMES = ["chr1", "chr10", "chr11", "chr12", "chr13", "chr14", "chr15", "chr16", "chr17", "chr18", "chr19", "chr2", "chr20", "chr21",
         "chr22", "chr3", "chr4", "chr5", "chr6", "chr7", "chr8", "chr9", "chrM", "chrX", "chrY"]
TYPES = ("VC", "VC_SQRT", "KR")


# ---------------------------------------------------------------- independent restatement
def bnewt(A, tol=1e-6, delta=0.1, Delta=3.0, etamax=0.1, g=0.9, max_outer=100):
    """Knight & Ruiz 2013, symmetric A with no empty row -> x with x * (A x) = 1, or None when it fails"""
    n = A.shape[0]
    x = np.ones(n); v = x * (A @ x); rk = 1 - v; rho_km1 = rk @ rk; rout = rold = rho_km1
    eta = etamax; rt = tol ** 2; stop_tol = 0.5 * tol; outer = 0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        while rout > rt:
            outer += 1
            if outer > max_outer:
                return None
            k = 0; y = np.ones(n); innertol = max(eta ** 2 * rout, rt)
            while rho_km1 > innertol:
                k += 1
                if k == 1:
                    Z = rk / v; p = Z.copy(); rho_km1 = rk @ Z
                else:
                    beta = rho_km1 / rho_km2; p = Z + beta * p
                w = x * (A @ (x * p)) + v * p
                alpha = rho_km1 / (p @ w); ap = alpha * p; ynew = y + ap
                if not np.isfinite(alpha):
                    return None
                if ynew.min() <= delta:
                    gamma = ((delta - y[ap < 0]) / ap[ap < 0]).min(); y = y + gamma * ap; break
                if ynew.max() >= Delta:
                    m = ynew > Delta
                    gamma = ((Delta - y[m]) / ap[m]).min(); y = y + gamma * ap; break
                y = ynew; rk = rk - alpha * w; rho_km2 = rho_km1; Z = rk / v; rho_km1 = rk @ Z
            x = x * y; v = x * (A @ x); rk = 1 - v; rho_km1 = rk @ rk; rout = rho_km1
            if not np.all(np.isfinite(x)) or x.min() <= 0 or not np.isfinite(rout):
                return None
            rat = rout / rold; rold = rout; eta_o = eta; eta = g * rat
            if g * eta_o ** 2 > 0.1:
                eta = max(eta, g * eta_o ** 2)
            eta = max(min(eta, etamax), stop_tol / np.sqrt(rout))
    return x


def chrom_parts(lens, res, b1, b2, ct):
    """per chromosome: (first bin, bins, upper-triangle intra entries x, y, c in chromosome coordinates)"""
    off = np.concatenate([[0], np.cumsum(np.array(lens, dtype=np.int64) // res + 1)])
    b1, b2, ct = (np.asarray(a, dtype=np.int64) for a in (b1, b2, ct))
    c1 = np.searchsorted(off, b1, side="right") - 1
    c2 = np.searchsorted(off, b2, side="right") - 1
    out = []
    for c in range(len(lens)):
        m = (c1 == c) & (c2 == c)
        out.append((int(off[c]), int(off[c + 1] - off[c]), b1[m] - off[c], b2[m] - off[c], ct[m].astype(np.float64)))
    return out


def sym(nb, x, y, c):
    U = sp.coo_matrix((c, (x, y)), shape=(nb, nb)).tocsr()
    return (U + U.T - sp.diags(U.diagonal())).tocsr()


def sum_factor(n, x, y, c):
    ok = np.isfinite(n[x]) & np.isfinite(n[y]) & (n[x] > 0) & (n[y] > 0)
    w = np.where(x != y, 2.0, 1.0)[ok]
    raw = (c[ok] * w).sum(); nrm = (c[ok] / (n[x[ok]] * n[y[ok]]) * w).sum()
    return n * np.sqrt(nrm / raw)


def ref_norms(lens, res, b1, b2, ct, types=TYPES):
    """-> ({type: vector over all bins}, status per chromosome) by the restatement"""
    nb_all = int(sum(l // res + 1 for l in lens))
    out = {t: np.zeros(nb_all) if t != "KR" else np.full(nb_all, np.nan) for t in types}
    status = []
    for o, nb, x, y, c in chrom_parts(lens, res, b1, b2, ct):
        if c.sum() == 0:
            status.append(1); continue
        A = sym(nb, x, y, c)
        rs = np.asarray(A.sum(axis=1)).ravel()
        st = 0
        if "VC" in types:
            out["VC"][o:o + nb] = sum_factor(rs.copy(), x, y, c)
        if "VC_SQRT" in types:
            out["VC_SQRT"][o:o + nb] = sum_factor(np.sqrt(rs), x, y, c)
        if "KR" in types:
            kept = rs > 0
            xk = bnewt(A[kept][:, kept])
            if xk is None:
                st = 2
            else:
                n = np.full(nb, np.nan); n[kept] = 1 / xk
                out["KR"][o:o + nb] = sum_factor(n, x, y, c)
        status.append(st)
    return out, status


# ---------------------------------------------------------------- GPU side
def gpu_coo(p, lens, res):
    n = len(p)
    d = to_dev(p)
    b1 = torch.empty(n + 1, dtype=torch.int32, device="cuda"); b2 = torch.empty_like(b1); ct = torch.empty_like(b1)
    ws = mk.PairsWorkspace(n + 1)
    nnz = ws.bin(d.data_ptr(), n, lens, res, b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), n + 1)
    ws.close()
    return b1, b2, ct, nnz


def gpu_norms(lens, res, b1, b2, ct, nnz, types=TYPES, max_nnz=None):
    nm = mk.Norm(lens, res, max_nnz if max_nnz is not None else max(nnz, 1))
    outs = {t: torch.full((nm.n_bins,), -1.0, dtype=torch.float64, device="cuda") for t in types}
    status, st = nm.run(b1.data_ptr(), b2.data_ptr(), ct.data_ptr(), nnz, types, **{("d_" + t.lower()): outs[t].data_ptr() for t in types})
    nm.close()
    return {t: v.cpu().numpy() for t, v in outs.items()}, status, st


def host(a, nnz):
    return a[:nnz].cpu().numpy().astype(np.uint32)


def toy_pairs(lens, n, seed, trans=0.2, skip=()):
    """power-law distance decay, a trans fraction; no pair touches the chromosomes in `skip` inside themselves"""
    rng = np.random.default_rng(seed)
    L = np.array(lens, dtype=np.int64)
    p = np.zeros(n, dtype=mk.PAIR_DTYPE)
    c1 = rng.choice(len(lens), n, p=L / L.sum())
    c2 = np.where(rng.random(n) < trans, rng.integers(0, len(lens), n), c1)
    for s in skip:
        c2 = np.where((c1 == s) & (c2 == s), (s + 1) % len(lens), c2)
    p1 = (rng.random(n) * (L[c1] - 1)).astype(np.int64) + 1
    d = np.exp(rng.random(n) * np.log(L.max())).astype(np.int64)
    p2 = np.where(c1 == c2, np.clip(p1 + d * rng.choice([-1, 1], n), 1, L[c2]), (rng.random(n) * (L[c2] - 1)).astype(np.int64) + 1)
    lo, hi = np.minimum(c1, c2), np.maximum(c1, c2)
    p["chr1"], p["chr2"] = lo, hi
    p["pos1"] = np.where(c1 <= c2, p1, p2); p["pos2"] = np.where(c1 <= c2, p2, p1)
    return p


def kr_properties(lens, res, b1, b2, ct, kr, status):
    """row sums of A / (n n^T) constant on kept rows; the normalised matrix sums to the raw one"""
    for c, (o, nb, x, y, cc) in enumerate(chrom_parts(lens, res, b1, b2, ct)):
        if status[c] != 0:
            continue
        A = sym(nb, x, y, cc)
        n = kr[o:o + nb]
        kept = np.isfinite(n)
        assert np.array_equal(kept, np.asarray(A.sum(axis=1)).ravel() > 0)
        inv = np.where(kept, 1 / np.where(kept, n, 1), 0)
        rows = inv * (A @ inv)
        assert np.ptp(rows[kept]) <= 1e-5 * rows[kept].mean(), (c, np.ptp(rows[kept]) / rows[kept].mean())
        w = np.where(x != y, 2.0, 1.0)
        assert np.isclose((cc * w / (n[x] * n[y])).sum(), (cc * w).sum(), rtol=1e-9)


# ---------------------------------------------------------------- tests
@pytest.mark.parametrize("res", [1000000, 100000])
def test_vc_hg38(res):
    p = random_pairs(300000, 21)
    b1, b2, ct, nnz = gpu_coo(p, HG38_LEN, res)
    got, status, _ = gpu_norms(HG38_LEN, res, b1, b2, ct, nnz, ("VC", "VC_SQRT"))
    exp, est = ref_norms(HG38_LEN, res, host(b1, nnz), host(b2, nnz), host(ct, nnz), ("VC", "VC_SQRT"))
    assert status == est
    for t in ("VC", "VC_SQRT"):
        np.testing.assert_allclose(got[t], exp[t], rtol=1e-12, atol=0)


def test_vc_and_kr_toy_genome():
    """a chromosome shorter than one bin, one without intra contacts (only trans pairs touch it)"""
    lens = [3000000, 2200000, 40000, 900000]
    p = toy_pairs(lens, 60000, 5, skip=(3,))
    res = 100000
    b1, b2, ct, nnz = gpu_coo(p, lens, res)
    got, status, st = gpu_norms(lens, res, b1, b2, ct, nnz)
    hb1, hb2, hct = host(b1, nnz), host(b2, nnz), host(ct, nnz)
    exp, est = ref_norms(lens, res, hb1, hb2, hct)
    assert status == est == [0, 0, 0, 1]
    for t in ("VC", "VC_SQRT"):
        np.testing.assert_allclose(got[t], exp[t], rtol=1e-12, atol=0)
    assert np.array_equal(np.isnan(got["KR"]), np.isnan(exp["KR"]))
    np.testing.assert_allclose(got["KR"], exp["KR"], rtol=1e-5)
    kr_properties(lens, res, hb1, hb2, hct, got["KR"], status)
    assert st.kr_failed == 0 and st.kr_residual_max <= 1e-6 and st.kr_matvecs > 0


def test_kr_hg38_1mb():
    p = random_pairs(400000, 22)
    res = 1000000
    b1, b2, ct, nnz = gpu_coo(p, HG38_LEN, res)
    got, status, st = gpu_norms(HG38_LEN, res, b1, b2, ct, nnz, ("KR",))
    hb1, hb2, hct = host(b1, nnz), host(b2, nnz), host(ct, nnz)
    exp, est = ref_norms(HG38_LEN, res, hb1, hb2, hct, ("KR",))
    assert status == est and 2 not in status
    assert np.array_equal(np.isnan(got["KR"]), np.isnan(exp["KR"]))
    np.testing.assert_allclose(got["KR"], exp["KR"], rtol=1e-5)
    kr_properties(HG38_LEN, res, hb1, hb2, hct, got["KR"], status)


def test_kr_failure_is_reported_and_isolated():
    """a 3-bin path (counts only at (0,1) and (1,2)) has no doubly-stochastic scaling; the other chromosomes of the call are
    bitwise what they are without it"""
    lens = [3000000, 250000, 1500000]
    res = 100000
    p = toy_pairs(lens, 40000, 9, trans=0.0, skip=(1,))
    b1, b2, ct, nnz = gpu_coo(p, lens, res)
    hb1, hb2, hct = host(b1, nnz), host(b2, nnz), host(ct, nnz)
    assert not ((hb1 >= 31) & (hb2 < 34)).any()                       # the middle chromosome has trans contacts only
    coo = sorted(list(zip(hb1.tolist(), hb2.tolist(), hct.tolist())) + [(31, 32, 5), (32, 33, 7)])
    d = [torch.tensor(np.array(a, dtype=np.uint32).view(np.int32), device="cuda") for a in zip(*coo)]
    got, status, st = gpu_norms(lens, res, *d, len(coo))
    assert status == [0, 2, 0] and st.kr_failed == 1
    assert np.isnan(got["KR"][31:34]).all() and (got["VC"][31:34] > 0).all()
    alone, status0, _ = gpu_norms(lens, res, b1, b2, ct, nnz)
    assert status0 == [0, 1, 0]
    for t in TYPES:
        keep = np.r_[0:31, 34:len(got[t])]
        assert got[t][keep].tobytes() == alone[t][keep].tobytes(), t
    exp, est = ref_norms(lens, res, *(np.array(a) for a in zip(*coo)))
    assert est == [0, 2, 0]


def test_bitwise_reproducible():
    p = random_pairs(300000, 23)
    res = 100000
    b1, b2, ct, nnz = gpu_coo(p, HG38_LEN, res)
    first, s1, _ = gpu_norms(HG38_LEN, res, b1, b2, ct, nnz)
    again, s2, _ = gpu_norms(HG38_LEN, res, b1, b2, ct, nnz)
    moved = [torch.empty(nnz + 977, dtype=torch.int32, device="cuda")[977:] for _ in range(3)]
    for m, a in zip(moved, (b1, b2, ct)):
        m.copy_(a[:nnz])
    other, s3, _ = gpu_norms(HG38_LEN, res, *moved, nnz)
    assert s1 == s2 == s3
    for t in TYPES:
        assert first[t].tobytes() == again[t].tobytes() == other[t].tobytes(), t


def test_hg38_5kb_lockstep():
    """>= 20 M pairs at 5 kb, all three types; KR against scipy on three chromosomes that converge at different steps"""
    p = random_pairs(20000000, 24, dup_frac=0.0)
    res = 5000
    b1, b2, ct, nnz = gpu_coo(p, HG38_LEN, res)
    got, status, st = gpu_norms(HG38_LEN, res, b1, b2, ct, nnz)
    hb1, hb2, hct = host(b1, nnz), host(b2, nnz), host(ct, nnz)
    parts = chrom_parts(HG38_LEN, res, hb1, hb2, hct)
    for c in (NAMES.index("chr19"), NAMES.index("chr21"), NAMES.index("chrM")):
        assert status[c] == 0
        o, nb, x, y, cc = parts[c]
        A = sym(nb, x, y, cc)
        rs = np.asarray(A.sum(axis=1)).ravel()
        np.testing.assert_allclose(got["VC"][o:o + nb], sum_factor(rs.copy(), x, y, cc), rtol=1e-12)
        np.testing.assert_allclose(got["VC_SQRT"][o:o + nb], sum_factor(np.sqrt(rs), x, y, cc), rtol=1e-12)
        kept = rs > 0
        xk = bnewt(A[kept][:, kept])
        n = np.full(nb, np.nan); n[kept] = 1 / xk
        n = sum_factor(n, x, y, cc)
        assert np.array_equal(np.isnan(got["KR"][o:o + nb]), np.isnan(n))
        np.testing.assert_allclose(got["KR"][o:o + nb], n, rtol=1e-5)
    assert st.kr_outer_max >= 2 and st.kr_residual_max <= 1e-6


def test_refusals():
    lens = [1000000, 500000]
    res = 100000                                                    # 11 + 6 bins
    ok = [torch.tensor(np.array(a, dtype=np.int32), device="cuda") for a in ([0, 1, 12], [1, 5, 16], [3, 4, 5])]
    nm = mk.Norm(lens, res, 2)
    outs = [torch.empty(17, dtype=torch.float64, device="cuda") for _ in TYPES]
    kw = dict(d_vc=outs[0].data_ptr(), d_vc_sqrt=outs[1].data_ptr(), d_kr=outs[2].data_ptr())
    with pytest.raises(mk.MkError, match="error -4"):
        nm.run(ok[0].data_ptr(), ok[1].data_ptr(), ok[2].data_ptr(), 3, TYPES, **kw)
    nm.close()
    nm = mk.Norm(lens, res, 3)
    status, _ = nm.run(ok[0].data_ptr(), ok[1].data_ptr(), ok[2].data_ptr(), 3, TYPES, **kw)
    assert status == [2, 0]                                         # bins 0 - 1 - 5 form a path: no KR scaling
    for bad in (([0, 1, 12], [1, 5, 17], [3, 4, 5]),                  # a bin past the end
                ([0, 5, 12], [1, 4, 16], [3, 4, 5])):                  # bin1 > bin2
        t = [torch.tensor(np.array(a, dtype=np.int32), device="cuda") for a in bad]
        with pytest.raises(mk.MkError, match="error -1"):
            nm.run(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), 3, TYPES, **kw)
    nm.close()
    with pytest.raises(mk.MkError, match="error -4"):
        mk.Norm(lens, res, 1 << 30)


# ---------------------------------------------------------------- pairs2bins -n
def run(cmd, **kw):
    return subprocess.run(cmd, capture_output=True, **kw)


def test_pairs2bins_norm_vectors(tmp_path):
    """dense (1 Mb, 100 kb), sort path (50 kb) and -d (5 kb) resolutions in one run; the file's vectors are byte-equal to
    mk_norm_device on the .coo the run wrote, and everything before the normalised section is the file of the same run without -n"""
    from hic_norm_reader import read_norm
    p = toy_pairs(HG38_LEN, 300000, 31)
    lines = [f"r{i}\t{NAMES[a]}\t{x}\t{NAMES[b]}\t{y}\t+\t-\n" for i, (a, x, b, y) in enumerate(zip(p["chr1"].tolist(), p["pos1"].tolist(), p["chr2"].tolist(), p["pos2"].tolist()))]
    pf = tmp_path / "x.pairs"; pf.write_text("## pairs format v1.0\n" + "".join(lines + lines[:5000]))
    info = tmp_path / "hg38.info"; info.write_text("".join(f"{n}\t{l}\n" for n, l in zip(NAMES, HG38_LEN)))
    res = [1000000, 100000, 50000, 5000]
    args = ["-r", ",".join(map(str, res)), str(pf)]
    r = run([os.path.join(BIN, "pairs2bins"), "-d", "-H", str(tmp_path / "n.hic"), "-n", "VC,VC_SQRT,KR"] + args + [str(tmp_path / "n"), str(info)])
    assert r.returncode == 0, r.stderr
    assert r.stderr.count(b"INFO: KR at ") == 4 and b"(2 dense)" in r.stderr
    r = run([os.path.join(BIN, "pairs2bins"), "-d", "-H", str(tmp_path / "p.hic")] + args + [str(tmp_path / "p"), str(info)])
    assert r.returncode == 0, r.stderr
    coo, norms = {}, {}
    for rs in res:
        text = (tmp_path / f"n.{rs}.coo").read_text()
        assert text == (tmp_path / f"p.{rs}.coo").read_text()
        a = np.loadtxt(tmp_path / f"n.{rs}.coo", dtype=np.int64, ndmin=2)
        coo[rs] = (a[:, 0], a[:, 1], a[:, 2])
        d = [torch.tensor(a[:, k].astype(np.int32), device="cuda") for k in range(3)]
        got, status, _ = gpu_norms(HG38_LEN, rs, *d, len(a))
        norms[rs] = {t: (got[t], [s != 1 if t != "KR" else s == 0 for s in status]) for t in TYPES}
    h = check_norm(str(tmp_path / "n.hic"), HG38_LEN, coo, norms)
    cut = h["section_start"]
    plain = (tmp_path / "p.hic").read_bytes()
    assert (tmp_path / "n.hic").read_bytes()[:cut] == plain[:cut] and plain[cut:] == b"\0" * 8
    assert read_norm(str(tmp_path / "p.hic"))["index"] == []


def test_pairs2bins_norm_usage(tmp_path):
    info = tmp_path / "g.info"; info.write_text("chr1\t1000\n")
    pf = tmp_path / "x.pairs"; pf.write_text("r\tchr1\t1\tchr1\t5\t+\t-\n")
    exe = os.path.join(BIN, "pairs2bins")
    assert run([exe, "-n", "VC", "-r", "100", str(pf), str(tmp_path / "o"), str(info)]).returncode == 2
    assert run([exe, "-H", str(tmp_path / "o.hic"), "-n", "FOO", "-r", "100", str(pf), str(tmp_path / "o"), str(info)]).returncode == 2
    assert run([exe, "-H", str(tmp_path / "o.hic"), "-n", "VC,KR,ICE", "-r", "100", str(pf), str(tmp_path / "o"), str(info)]).returncode == 2
