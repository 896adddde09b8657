"""Normalisation vectors in the `.hic` writer (csrc/hic_writer.hpp, host-only): a small harness compiled here hands the writer COO
triplets with given vectors, and the file is read back with the independent tests/hic_norm_reader.py.  Without vectors the file is
byte-identical to bin/coo2hic's, and with them everything in front of the normalised section is unchanged."""
import os
import struct
import subprocess

import numpy as np
import pytest

from hic_norm_check import check_norm
from test_hic_writer import contacts, coo, write_coo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "microcket_b200", "csrc")
COO2HIC = os.path.join(ROOT, "microcket_b200", "bin", "coo2hic")

HARNESS = r"""
#include "hic_writer.hpp"
#include <fstream>
#include <iostream>
// harness <genome> <info> <out.hic> <spec>; spec lines: "R <res> <coo.bin>" (u64 nnz, u32 bin1[nnz], bin2[nnz], count[nnz]), then
// for that resolution any number of "N <type> <values.bin> <stored.bin>" (f64 per bin, u8 per chromosome)
template <class T> static std::vector<T> slurp(const std::string &p) {
    std::ifstream f(p, std::ios::binary); std::vector<char> b((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    std::vector<T> v(b.size() / sizeof(T)); memcpy(v.data(), b.data(), v.size() * sizeof(T)); return v;
}
int main(int argc, char **argv) {
    if (argc != 5) return 2;
    std::vector<std::string> names; std::vector<uint32_t> lens;
    { std::ifstream fi(argv[2]); std::string n; uint32_t l; while (fi >> n >> l) { names.push_back(n); lens.push_back(l); } }
    struct R { uint32_t res; std::string coo; std::vector<std::string> t, v, s; };
    std::vector<R> rs;
    { std::ifstream fs(argv[4]); std::string k; while (fs >> k) {
        if (k == "R") { rs.emplace_back(); fs >> rs.back().res >> rs.back().coo; }
        else { std::string a, b, c; fs >> a >> b >> c; rs.back().t.push_back(a); rs.back().v.push_back(b); rs.back().s.push_back(c); } } }
    std::vector<uint32_t> res; for (auto &r : rs) res.push_back(r.res);
    hic::Writer w(argv[1], names, lens, res);
    std::string err;
    for (auto &r : rs) {
        std::vector<uint32_t> c = slurp<uint32_t>(r.coo);
        const size_t n = (size_t)c[0] | ((size_t)c[1] << 32);
        std::vector<std::vector<double>> vals; std::vector<hic::NormInput> norms;
        for (size_t k = 0; k < r.t.size(); ++k) vals.push_back(slurp<double>(r.v[k]));
        for (size_t k = 0; k < r.t.size(); ++k) {
            std::vector<uint8_t> st = slurp<uint8_t>(r.s[k]);
            hic::NormInput q; q.type = r.t[k]; q.values = vals[k].data(); q.stored.assign(st.begin(), st.end()); norms.push_back(q);
        }
        if (w.add(r.res, c.data() + 2, c.data() + 2 + n, c.data() + 2 + 2 * n, n, &err, r.t.empty() ? nullptr : &norms)) { std::cerr << err << "\n"; return 10; }
    }
    if (w.write(argv[3], &err)) { std::cerr << err << "\n"; return 10; }
    return 0;
}
"""

NAMES = ["chr1", "chr10", "chr2", "chrM", "chrX", "chrEmpty"]
LENS = [24895642, 13379742, 9000001, 16569, 4999999, 700000]


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("harness")
    (d / "h.cpp").write_text(HARNESS)
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", CSRC, "-o", str(d / "h"), str(d / "h.cpp"), "-lz", "-pthread"], check=True)
    subprocess.run(["make", "-C", CSRC, "../bin/coo2hic"], check=True, capture_output=True)
    return str(d / "h")


def vectors(rng, lens, res, stored):
    """positive values with NaN and zero entries sprinkled in, over all bins"""
    nb = int(sum(l // res + 1 for l in lens))
    v = rng.random(nb) * 2 + 0.05
    v[rng.random(nb) < 0.02] = np.nan
    v[rng.random(nb) < 0.02] = 0.0
    return v, stored


def run(harness, tmp_path, by_res, norms_by_res, name):
    info = tmp_path / "toy.info"
    info.write_text("".join(f"{n}\t{l}\n" for n, l in zip(NAMES, LENS)))
    spec = []
    for res, (b1, b2, ct) in by_res.items():
        f = tmp_path / f"{name}.{res}.coo.bin"
        f.write_bytes(struct.pack("<Q", len(b1)) + b"".join(np.asarray(a, dtype="<u4").tobytes() for a in (b1, b2, ct)))
        spec.append(f"R {res} {f}")
        for typ, (vals, stored) in norms_by_res.get(res, {}).items():
            fv = tmp_path / f"{name}.{res}.{typ}.f64"; fv.write_bytes(np.asarray(vals, dtype="<f8").tobytes())
            fs = tmp_path / f"{name}.{res}.{typ}.u8"; fs.write_bytes(np.asarray(stored, dtype=np.uint8).tobytes())
            spec.append(f"N {typ} {fv} {fs}")
    (tmp_path / f"{name}.spec").write_text("\n".join(spec) + "\n")
    out = tmp_path / f"{name}.hic"
    r = subprocess.run([harness, "toy", str(info), str(out), str(tmp_path / f"{name}.spec")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return out


def test_vectors_and_normalised_expected_values_read_back(harness, tmp_path):
    c1, p1, c2, p2 = contacts(LENS[:5], 200000, 11)
    by_res = {r: coo(LENS, r, c1, p1, c2, p2) for r in (1000000, 50000, 5000)}
    rng = np.random.default_rng(3)
    stored_all = [True, True, True, True, True, False]              # chrEmpty: no intra contacts, no vector
    stored_kr = [True, False, True, True, True, False]              # chr10's KR "failed"
    norms = {1000000: {"VC": vectors(rng, LENS, 1000000, stored_all), "KR": vectors(rng, LENS, 1000000, stored_kr)},
             50000: {"VC": vectors(rng, LENS, 50000, stored_all), "VC_SQRT": vectors(rng, LENS, 50000, stored_all),
                     "KR": vectors(rng, LENS, 50000, stored_kr)},
             5000: {"KR": vectors(rng, LENS, 5000, stored_kr)}}
    with_v = run(harness, tmp_path, by_res, norms, "with")
    h = check_norm(str(with_v), LENS, by_res, norms)
    assert len(h["vectors"]) == 5 + 4 + 5 + 5 + 4 + 4 and ("KR", 2, 5000) not in h["vectors"]
    assert ("KR", 5000) in h["expected"] and ("VC_SQRT", 50000) in h["expected"]
    # no vectors: byte-identical to coo2hic; with vectors: identical up to the end of the raw footer
    none = run(harness, tmp_path, by_res, {}, "none")
    for res, (b1, b2, ct) in by_res.items():
        write_coo(str(tmp_path / "in"), res, b1, b2, ct)
    info = tmp_path / "toy.info"
    r = subprocess.run([COO2HIC, "-g", "toy", "-r", ",".join(map(str, by_res)), str(tmp_path / "in"), str(tmp_path / "c.hic"), str(info)], capture_output=True)
    assert r.returncode == 0, r.stderr
    plain = (tmp_path / "c.hic").read_bytes()
    assert none.read_bytes() == plain
    cut = h["section_start"]
    assert with_v.read_bytes()[:cut] == plain[:cut] and plain[cut:] == struct.pack("<ii", 0, 0)


def test_a_resolution_without_vectors_and_a_type_without_valid_entries(harness, tmp_path):
    names_lens = LENS
    c1, p1, c2, p2 = contacts(names_lens[:5], 30000, 12)
    by_res = {r: coo(names_lens, r, c1, p1, c2, p2) for r in (2500000, 100000)}
    nb = int(sum(l // 100000 + 1 for l in names_lens))
    nan = np.full(nb, np.nan)                                        # every norm invalid: vectors stored, no expected values
    norms = {100000: {"KR": (nan, [True] * 5 + [False])}}
    out = run(harness, tmp_path, by_res, norms, "x")
    h = check_norm(str(out), names_lens, by_res, norms)
    assert ("KR", 100000) not in h["expected"] and len(h["vectors"]) == 5
