"""SAM -> coordinate-sorted BAM + .bai on the GPU (csrc/bam_out.cu, bin/sam2bam).  The device encoder against
tests/bam_writer.encode_records, the sort against numpy's stable lexsort, and the executable's output read back by gzip, by
bin/bam2sam and, for the index, by tests/bai_reader.py: counts, chunks at record starts of their bin, a linear index that is a
lower bound, and region queries equal to a brute-force overlap.  Spilled runs and merge rounds give the in-core bytes."""
import gzip
import os
import struct
import subprocess

import numpy as np
import pytest

import microcket_b200 as mk
import bam_corpus as BC
import bai_reader as BR

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
BIN = os.path.join(os.path.dirname(mk.LIB_PATH), "bin")
SAM2BAM, BAM2SAM = os.path.join(BIN, "sam2bam"), os.path.join(BIN, "bam2sam")
HG38 = list(zip(["chr1", "chr10", "chr11", "chr12", "chr13", "chr14", "chr15", "chr16", "chr17", "chr18", "chr19", "chr2", "chr20", "chr21",
                 "chr22", "chr3", "chr4", "chr5", "chr6", "chr7", "chr8", "chr9", "chrM", "chrX", "chrY"],
                [248956422, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616,
                 242193529, 64444167, 46709983, 50818468, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717,
                 16569, 156040895, 57227415]))
ALL = HG38 + [("scaffold_7", 40000)]


def dev(data):
    return torch.frombuffer(bytearray(data) + bytearray(16), dtype=torch.uint8).to("cuda")


def encode_device(bam, text, cuts):
    """text encoded in calls cut at the given line indices -> (record bytes, offsets)"""
    lines = text.splitlines(keepends=True)
    cap = 4 * len(text) + 1024
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    off = torch.zeros(len(lines) + 1, dtype=torch.int64, device="cuda")
    base, n = 0, 0
    for a, b in zip([0] + cuts, cuts + [len(lines)]):
        part = "".join(lines[a:b]).encode()
        if not part:
            continue
        d = dev(part)
        nl, rb = bam.encode(d.data_ptr(), len(part), out.data_ptr(), cap, off.data_ptr() + 8 * n, base)
        assert nl == b - a
        base += rb; n += nl
    torch.cuda.synchronize()
    return out, off, n, base


def test_device_encode_equals_bam_writer():
    exp = BC.expected_records(BC.CORPUS)
    bam = mk.Bam(BC.REFS, 1 << 20, 4096)
    nlines = len(BC.CORPUS.splitlines())
    for cuts in ([], [1], [3, 9], list(range(1, nlines))):
        out, off, n, nb = encode_device(bam, BC.CORPUS, cuts)
        assert out[:nb].cpu().numpy().tobytes() == exp, cuts
        o = off[:n + 1].cpu().numpy()
        assert o[0] == 0 and o[-1] == nb and [int(x) for x in np.diff(o)] == [len(r) for r in BC.split_records(exp)]
    bam.close()


def test_device_refusals_name_the_line():
    bam = mk.Bam(BC.REFS, 1 << 20, 4096)
    good = BC.CORPUS.splitlines()
    out = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    off = torch.empty(4096, dtype=torch.int64, device="cuda")
    for k, (bad, code) in enumerate(BC.REFUSALS):
        at = (7 * k) % (len(good) + 1)
        lines = good[:at] + [bad] + good[at:] + [BC.REFUSALS[(k + 1) % len(BC.REFUSALS)][0]]
        t = ("\n".join(lines) + "\n").encode()
        with pytest.raises(mk.BamInputError) as e:
            bam.encode(dev(t).data_ptr(), len(t), out.data_ptr(), 1 << 20, off.data_ptr())
        assert (e.value.line, e.value.code) == (at, code), bad[:60]
    bam.close()


def synth_text(n=20000, seed=3):
    flash = mk.synth_host(seed, "flash", "hg38", 0, n, mk.synth_opts(dup_per_1024=150, dup_universe=n)).decode()
    unc = mk.synth_host(seed + 1, "unc", "hg38", 0, n, mk.synth_opts(dup_per_1024=150, dup_universe=n)).decode()
    return flash + unc


def test_sort_equals_stable_lexsort():
    text = synth_text(6000) + BC.CORPUS
    exp = BC.sorted_records(BC.expected_records(text, ALL), len(ALL))
    lines = len(text.splitlines())
    bam = mk.Bam(ALL, len(text) + 16, lines + 16)
    out, off, n, nb = encode_device(bam, text, [lines // 3, lines // 2])
    assert bam.sort(out.data_ptr(), off.data_ptr(), n) == nb
    dst = torch.empty(nb + 16, dtype=torch.uint8, device="cuda")
    got, i0, u = [], 0, 0
    while i0 < n:                                          # slices of about 100 kB
        i1, b, _ = bam.gather(i0, 100000, dst.data_ptr() + u, nb + 16 - u)
        u += b; i0 = i1
    assert u == nb
    assert BC.split_records(dst[:nb].cpu().numpy().tobytes()) == exp
    bam.close()


def run(args, inp=None, env=None, **kw):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([SAM2BAM] + args, input=inp, capture_output=True, env=e, **kw)


def canonical(text):
    """RNEXT written '=' where it equals RNAME (what bam2sam prints)"""
    out = []
    for ln in text.splitlines():
        f = ln.split("\t")
        if f[6] == f[2] and f[2] != "*":
            f[6] = "="
        out.append("\t".join(f))
    return "\n".join(out) + "\n"


def check_bam(path, text, refs, hd_first=None):
    data = open(path, "rb").read()
    assert data.endswith(mk.BGZF_EOF)
    raw = gzip.decompress(data)
    f = BR.BamFile(data)
    assert max(f.isizes) <= 65280
    assert f.refs == [(n, l) for n, l in refs]
    first = f.text.split("\n")[0]
    assert first == (hd_first or "@HD\tVN:1.6\tSO:coordinate")
    exp = BC.sorted_records(BC.expected_records(text, refs), len(refs))
    assert [r for _, r in f.records] == exp
    assert raw[f.rec_start:] == b"".join(exp)
    # the record stream starts at a member boundary
    assert f.rec_start in f.uoff
    return f


def check_bai(f, bai_bytes, n_ref, rng):
    idx = BR.parse(bai_bytes)
    assert len(idx["refs"]) == n_ref
    for order in BR.bin_order(bai_bytes):
        assert order == sorted(order)
    fields = [BR.rec_fields(r) for _, r in f.records]
    assert idx["n_no_coor"] == sum(1 for t, *_ in fields if t < 0)
    for t in range(n_ref):
        r = idx["refs"][t]
        mine = [k for k, x in enumerate(fields) if x[0] == t]
        if not mine:
            assert r["pseudo"] is None and not r["bins"] and not r["linear"]
            continue
        ps = r["pseudo"]
        assert ps["n_mapped"] == sum(1 for k in mine if not fields[k][4] & 4)
        assert ps["n_unmapped"] == sum(1 for k in mine if fields[k][4] & 4)
        assert f.resolve(ps["beg"]) == f.records[mine[0]][0]
        last = f.records[mine[-1]]
        assert f.resolve(ps["end"]) == last[0] + len(last[1])
        for b, chunks in r["bins"].items():                        # chunks start at records of their bin, hold only those
            for c in chunks:
                ks = f.records_in(c)
                assert ks and all(fields[k][0] == t and fields[k][3] == b for k in ks)
        covered = sorted(k for chunks in r["bins"].values() for c in chunks for k in f.records_in(c))
        assert covered == mine
        max_end = max(fields[k][2] for k in mine)
        assert len(r["linear"]) == (max_end - 1 >> 14) + 1
        first = {}                                                  # window -> the first record overlapping it
        for k in mine:
            for w in range(fields[k][1] >> 14, (max(fields[k][2] - 1, 0) >> 14) + 1):
                first.setdefault(w, k)
        for w, v in enumerate(r["linear"]):                         # a lower bound, exact where the window has records
            if w in first:
                assert f.resolve(v) == f.records[first[w]][0]
        pos = np.array([fields[k][1] for k in mine]); end_ = np.array([fields[k][2] for k in mine]); ks = np.array(mine)
        L = max_end + 20000
        for _ in range(120):                                       # region queries against brute force
            beg = int(rng.integers(0, L)); end = beg + int(rng.integers(1, 300000))
            hits = {k for c in BR.query_chunks(idx, t, beg, end) for k in f.records_in(c)
                    if fields[k][0] == t and fields[k][1] < end and fields[k][2] > beg}
            brute = set(ks[(pos < end) & (end_ > beg)].tolist())
            assert hits == brute, (t, beg, end)
    return idx


@pytest.fixture(scope="module")
def sam(tmp_path_factory):
    d = tmp_path_factory.mktemp("sam2bam")
    text = synth_text(20000) + BC.CORPUS
    hdr = BC.header(ALL)
    p = d / "in.sam"
    p.write_text(hdr + text)
    return d, hdr, text


def test_sam2bam_in_core(sam):
    d, hdr, text = sam
    r = run(["-o", str(d / "a.bam"), str(d / "in.sam")])
    assert r.returncode == 0, r.stderr
    assert b"INFO" in r.stderr and b"0 runs spilled, 0 merge rounds" in r.stderr
    f = check_bam(d / "a.bam", text, ALL, "@HD\tVN:1.6\tSO:coordinate")
    check_bai(f, open(str(d / "a.bam") + ".bai", "rb").read(), len(ALL), np.random.default_rng(0))
    assert not [x for x in os.listdir(d) if ".tmp." in x]


def test_sam2bam_bam2sam_prints_sorted_input(tmp_path):
    text = synth_text(3000, seed=9)
    p = tmp_path / "s.sam"
    p.write_text(BC.header(HG38, hd=None) + text)
    assert run(["-o", str(tmp_path / "s.bam"), str(p)]).returncode == 0
    lines = canonical(text).splitlines()
    recs = BC.expected_records("\n".join(lines) + "\n", HG38)
    keys = np.array([BC.sort_key(r, len(HG38)) for r in BC.split_records(recs)], dtype=np.int64)
    order = np.lexsort((keys[:, 2], keys[:, 1], keys[:, 0]))
    out = subprocess.run([BAM2SAM, str(tmp_path / "s.bam")], capture_output=True, check=True).stdout.decode()
    body = [ln for ln in out.splitlines() if not ln.startswith("@")]
    assert body == [lines[k] for k in order]


def test_sam2bam_spills_give_the_same_bytes(sam):
    d, hdr, text = sam
    assert run(["-o", str(d / "a.bam"), str(d / "in.sam")]).returncode == 0
    r = run(["-o", str(d / "b.bam"), str(d / "in.sam")], env={"MICROCKET_CHUNK_MB": "1", "MICROCKET_SORT_MB": "4"})
    assert r.returncode == 0, r.stderr
    info = r.stderr.decode().split("INFO: ")[1].split()
    spilled, rounds = int(info[2]), int(info[5])
    assert spilled >= 5 and rounds >= 3, r.stderr
    assert open(d / "b.bam", "rb").read() == open(d / "a.bam", "rb").read()
    assert open(str(d / "b.bam") + ".bai", "rb").read() == open(str(d / "a.bam") + ".bai", "rb").read()
    assert not [x for x in os.listdir(d) if ".tmp." in x]


def test_sam2bam_files_equal_stdin(sam):
    d, hdr, text = sam
    lines = text.splitlines(keepends=True)
    parts = [hdr, "".join(lines[:len(lines) // 3]), "".join(lines[len(lines) // 3:])]
    names = []
    for k, p in enumerate(parts):
        (d / f"p{k}.sam").write_text(p); names.append(str(d / f"p{k}.sam"))
    assert run(["-o", str(d / "m.bam")] + names).returncode == 0
    assert run(["-o", str(d / "s.bam"), "-"], inp=(hdr + text).encode()).returncode == 0
    assert run(["-o", str(d / "n.bam")], inp=(hdr + text).encode()).returncode == 0
    for x in ("m.bam", "n.bam"):
        assert open(d / x, "rb").read() == open(d / "s.bam", "rb").read()
        assert open(str(d / x) + ".bai", "rb").read() == open(str(d / "s.bam") + ".bai", "rb").read()


def test_sam2bam_empty_and_unmapped(tmp_path):
    r = run(["-o", str(tmp_path / "e.bam")], inp=b"")
    assert r.returncode == 0, r.stderr
    f = BR.BamFile(open(tmp_path / "e.bam", "rb").read())
    assert f.text == "@HD\tVN:1.6\tSO:coordinate\n" and f.refs == [] and f.records == []
    assert open(str(tmp_path / "e.bam") + ".bai", "rb").read() == b"BAI\1" + struct.pack("<iQ", 0, 0)
    text = "".join(f"u{k}\t4\t*\t0\t0\t*\t*\t0\t0\tACGT\tIIII\n" for k in range(5000))
    hdr = BC.header(BC.REFS, hd="@HD\tVN:1.4")
    (tmp_path / "u.sam").write_text(hdr + text)
    assert run(["-o", str(tmp_path / "u.bam"), str(tmp_path / "u.sam")]).returncode == 0
    f = check_bam(tmp_path / "u.bam", text, BC.REFS, "@HD\tVN:1.4\tSO:coordinate")
    idx = BR.parse(open(str(tmp_path / "u.bam") + ".bai", "rb").read())
    assert idx["n_no_coor"] == 5000 and all(r["pseudo"] is None for r in idx["refs"])


@pytest.mark.parametrize("case", ["bad_line", "late_header", "dup_sq", "no_ln", "unknown_ref", "missing_input"])
def test_sam2bam_refusals(tmp_path, case):
    good = BC.CORPUS
    hdr = BC.header(BC.REFS)
    body, expect = {
        "bad_line": (hdr + good + "x\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\n", f"line {len(hdr.splitlines()) + len(good.splitlines()) + 1}:"),
        "late_header": (hdr + good + "@CO\tlate\n", f"line {len(hdr.splitlines()) + len(good.splitlines()) + 1}:"),
        "dup_sq": (hdr + "@SQ\tSN:chr1\tLN:5\n" + good, "twice"),
        "no_ln": ("@SQ\tSN:chr1\n" + good, "no LN"),
        "unknown_ref": (BC.header(BC.REFS[:2]) + good, "not in @SQ"),
        "missing_input": ("", "cannot read"),
    }[case]
    p = tmp_path / "in.sam"
    if case != "missing_input":
        p.write_text(body)
    out = tmp_path / "o.bam"
    r = run(["-o", str(out), str(p)], env={"MICROCKET_CHUNK_MB": "1", "MICROCKET_SORT_MB": "4"})
    assert r.returncode == 10, r.stderr
    assert expect in r.stderr.decode(), r.stderr
    assert sorted(os.listdir(tmp_path)) == ([] if case == "missing_input" else ["in.sam"])
