"""BGZF deflate without a GPU: the host form of the member encoder (csrc/bgzf_deflate.h, the per-member decisions the kernel makes,
through tests/bgzf_deflate_host.cpp) built with AddressSanitizer and UBSan, its output read back by Python's zlib and gzip; code
lengths on adversarial histograms; and the option refusals of `bgzip`, which come before any device call."""
import gzip
import os
import shutil
import subprocess
import zlib

import numpy as np
import pytest

import microcket_b200 as mk
import bgzf_corpus as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BGZIP = os.path.join(os.path.dirname(mk.LIB_PATH), "bin", "bgzip")
HEADER = bytes.fromhex("1f8b08040000000000ff060042430200")


def sorted_text(text):
    lines = text.split(b"\n")
    hdr, body = lines[:2], [ln for ln in lines[2:] if ln]
    return b"\n".join(hdr + sorted(body, key=lambda ln: (ln.split(b"\t")[1], int(ln.split(b"\t")[2])))) + b"\n"


def inputs(seed=0):
    """name -> bytes: the lengths around the member cut, .pairs text in both orders, random bytes, runs and periods"""
    rng = np.random.default_rng(seed)
    text = B.pairs_text(30000, seed)
    out = {f"len{n}": text[:n] for n in (0, 1, 3, 4, 257, 258, 259, 65279, 65280, 65281, 2 * 65280)}
    out["pairs"] = text
    out["pairs_sorted"] = sorted_text(text)
    out["random"] = rng.integers(0, 256, 3 * 65280 + 99, dtype=np.uint8).tobytes()
    out["one_byte"] = b"A" * 200000
    for p in (1, 2, 3, 32768, 32769):
        unit = rng.integers(0, 256, p, dtype=np.uint8).tobytes()
        out[f"period{p}"] = (unit * (150000 // p + 2))[:150000]
    out["all_bytes"] = bytes(range(256)) * 300
    return out


def check_members(blob, data):
    """the member walk, bgzip's header bytes, member k = input slice k, each member alone inflated by raw zlib"""
    mem = B.members(blob)
    assert len(mem) == -(-len(data) // B.BLOCK)
    for k, (o, n, isize) in enumerate(mem):
        m = blob[o:o + n]
        assert n <= 65536 and m[:16] == HEADER and int.from_bytes(m[16:18], "little") == n - 1
        assert zlib.decompress(m[18:-8], -15) == data[k * B.BLOCK:(k + 1) * B.BLOCK]
    assert gzip.decompress(blob + B.EOF) == data
    return mem


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("bgzf_deflate_host")
    exe = d / "bgzf_deflate_host"
    cmd = [cxx, "-std=c++17", "-g", "-O1", "-Wall", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
           "-I", os.path.join(ROOT, "microcket_b200", "csrc"), os.path.join(ROOT, "tests", "bgzf_deflate_host.cpp"), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe), d


def host_compress(host, data, level=-1):
    exe, d = host
    (d / "in").write_bytes(data)
    r = subprocess.run([exe, "c", str(level), str(d / "in"), str(d / "out")], capture_output=True, text=True)
    assert r.returncode == 0 and "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-3000:]
    return (d / "out").read_bytes()


def test_host_form_round_trips_through_zlib(host):
    for name, data in inputs().items():
        blob = host_compress(host, data)
        check_members(blob, data)
        assert blob == host_compress(host, data, level=9), name         # every level but 0 writes the same bytes


def test_host_form_stored_members(host):
    data = inputs()["random"]
    for level in (0, -1):                                                # random bytes: every member stored either way
        blob = host_compress(host, data, level)
        for o, n, isize in check_members(blob, data):
            assert blob[o + 18] == 1 and n == isize + 31
    text = inputs()["pairs"]
    assert all(n == i + 31 for _, n, i in check_members(host_compress(host, text, 0), text))


def test_host_form_is_no_larger_than_zlib_level_1(host):
    text = B.pairs_text(300_000, seed=3)
    for data in (text, sorted_text(text)):
        z1 = sum(len(B.member(data[p:p + B.BLOCK], level=1)) for p in range(0, len(data), B.BLOCK))
        assert len(host_compress(host, data)) <= z1


def lengths(host, rows):
    exe, _ = host
    r = subprocess.run([exe, "h"], input="".join(f"{m} " + " ".join(map(str, f)) + "\n" for m, f in rows), capture_output=True, text=True)
    assert r.returncode == 0 and "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-3000:]
    return [list(map(int, ln.split())) for ln in r.stdout.splitlines()]


def test_code_lengths_on_adversarial_histograms(host):
    fib = [1, 1]
    while len(fib) < 30:
        fib.append(fib[-1] + fib[-2])
    rng = np.random.default_rng(5)
    rows = [(15, fib + [0] * 256), (15, [0] * 256 + fib), (7, fib[:19]), (15, [0] * 100 + [7] + [0] * 185), (15, [0] * 286),
            (15, [0] * 40 + [3] + [0] * 200 + [9] + [0] * 44), (15, [1] * 286), (7, [5] * 19), (7, [0] * 18 + [1]),
            (15, rng.integers(0, 65281, 286).tolist()), (15, (rng.integers(0, 2, 286) * rng.integers(1, 50, 286)).tolist())]
    for (maxlen, f), ln in zip(rows, lengths(host, rows)):
        assert len(ln) == len(f) and max(ln) <= maxlen
        used = [i for i, c in enumerate(f) if c]
        assert all(ln[i] for i in used)                                  # every counted symbol has a code
        assert sum(1 for x in ln if x) >= 2                              # at least two codes ...
        assert sum(2.0 ** -x for x in ln if x) == 1.0                    # ... and a complete one
        for i in used:                                                   # a more frequent symbol never has a longer code
            for j in used:
                assert f[i] <= f[j] or ln[i] <= ln[j]
    assert huffman_depth(fib) > 15                                       # the Fibonacci counts do need the limit


def huffman_depth(f):
    """the longest code of an unconstrained Huffman code of the counts f"""
    import heapq
    h = [(c, 0) for c in f if c]
    heapq.heapify(h)
    while len(h) > 1:
        a, b = heapq.heappop(h), heapq.heappop(h)
        heapq.heappush(h, (a[0] + b[0], max(a[1], b[1]) + 1))
    return h[0][1]


def test_bound():
    assert [mk.bgzf_deflate_bound(n) for n in (0, 1, 65280, 65281)] == [0, 32, 65311, 65281 + 62]


def test_bgzip_refuses_other_options(tmp_path):
    f = tmp_path / "x"
    f.write_bytes(b"a\n")
    for args in (["-i"], ["-b", "0"], ["-s", "5"], ["-r"], ["--index"], ["-l", "10"], ["-l"], ["-@"], [str(f), str(f)]):
        r = subprocess.run([BGZIP] + args + [str(f)], capture_output=True, text=True)
        assert r.returncode == 2 and "Usage:" in r.stderr and "Exit codes" in r.stderr, (args, r.stderr)
    assert f.read_bytes() == b"a\n" and not (tmp_path / "x.gz").exists()
    r = subprocess.run([BGZIP, "-h"], capture_output=True, text=True)
    assert r.returncode == 0 and "Usage:" in r.stderr
