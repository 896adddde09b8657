"""Shared by tests/test_hic_norm_writer.py (CPU, the writer through a harness) and tests/test_gpu_norm.py (`pairs2bins -n`): the
normalised section of a `.hic`, read back with tests/hic_norm_reader.py, must hold exactly the vectors it was given and normalised
expected values that satisfy their defining sums on the normalised counts."""
import numpy as np

from hic_norm_reader import read_norm


def valid_norm(v):
    return np.isfinite(v) & (v > 0)


def check_norm(path, lens, coo_by_res, norms_by_res):
    """coo_by_res: {res: (bin1, bin2, count)}, global bins; norms_by_res: {res: {type: (values over all bins, stored per chromosome)}}"""
    h = read_norm(path)
    lens = np.array(lens, dtype=np.int64)
    n = len(lens)
    assert [ln for _, ln in h["chroms"][1:]] == lens.tolist()
    want = set()
    for res, by_type in norms_by_res.items():
        off = np.concatenate([[0], np.cumsum(lens // res + 1)])
        b1, b2, ct = (np.asarray(a, dtype=np.int64) for a in coo_by_res[res])
        c1 = np.searchsorted(off, b1, side="right") - 1
        c2 = np.searchsorted(off, b2, side="right") - 1
        intra = c1 == c2
        for typ, (vals, stored) in by_type.items():
            vals = np.asarray(vals, dtype=np.float64)
            assert len(vals) == off[-1]
            for c in range(n):
                key = (typ, c + 1, res)
                if not stored[c]:
                    assert key not in h["vectors"], key
                    continue
                want.add(key)
                got = np.array(h["vectors"][key], dtype=np.float64)
                assert len(got) == lens[c] // res + 1
                assert got.tobytes() == vals[off[c]:off[c + 1]].tobytes(), key      # byte-equal, NaN included
            # normalised expected values: the raw procedure's sums, on c / (n_x n_y) of the entries with two valid norms
            ok_chr = np.array(stored, dtype=bool)
            m = intra & ok_chr[c1] & valid_norm(vals[b1]) & valid_norm(vals[b2])
            if not m.any():
                assert (typ, res) not in h["expected"]
                continue
            w = ct[m] / (vals[b1[m]] * vals[b2[m]])
            dist = (b2 - b1)[m]
            obs = np.bincount(c1[m], weights=w, minlength=n)
            ev, scale = h["expected"][(typ, res)]
            ev = np.array(ev)
            assert len(ev) == dist.max() + 1 and (ev >= 0).all() and ev[-1] > 0
            assert sorted(scale) == [int(k) + 1 for k in np.nonzero(obs > 0)[0]]
            for k, s in scale.items():
                nb = int(lens[k - 1] // res + 1)
                d = np.arange(min(nb, len(ev)))
                assert np.isclose((ev[d] * (nb - d)).sum(), s * obs[k - 1], rtol=1e-9)
            actual = np.bincount(dist, weights=w)
            possible = np.zeros(len(actual))
            for k in np.nonzero(obs > 0)[0]:
                nb = int(lens[k] // res + 1)
                d = np.arange(min(nb, len(actual)))
                possible[d] += nb - d
            if actual[0] >= 400:                                    # no smoothing window opens for the diagonal: a plain average
                assert np.isclose(ev[0], actual[0] / possible[0], rtol=1e-12)
    assert set(h["vectors"]) == want
    assert all(1 <= ci <= n for _, ci, _ in h["vectors"])
    assert set(h["expected"]) <= {(t, r) for r, bt in norms_by_res.items() for t in bt}
    return h
