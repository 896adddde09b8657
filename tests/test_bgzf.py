"""BGZF inflate without a GPU: the host form of the member decoder (csrc/bgzf_member.h, the control logic the kernel runs, through
tests/bgzf_host.cpp) built with AddressSanitizer and UBSan, against Python's zlib as an independent oracle, on well-formed and
damaged members; and the library's host member walk (mk_bgzf_scan)."""
import gzip
import os
import shutil
import struct
import subprocess
import zlib

import pytest

import microcket_b200 as mk
import bgzf_corpus as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("bgzf_host")
    exe = d / "bgzf_host"
    cmd = [cxx, "-std=c++17", "-g", "-O1", "-Wall", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
           "-I", os.path.join(ROOT, "microcket_b200", "csrc"), os.path.join(ROOT, "tests", "bgzf_host.cpp"), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe), d


def run_host(host, blobs):
    """-> [(status line, output bytes or None)] of the host decoder on each BGZF byte string; fails on any sanitizer report"""
    exe, d = host
    res = []
    for b0 in range(0, len(blobs), 2000):
        files = []
        for k, blob in enumerate(blobs[b0:b0 + 2000]):
            f = d / f"in{k}"
            f.write_bytes(blob)
            if os.path.exists(str(f) + ".out"):
                os.remove(str(f) + ".out")
            files.append(str(f))
        r = subprocess.run([exe] + files, capture_output=True, text=True, env={**os.environ, "ASAN_OPTIONS": "detect_leaks=1"})
        assert r.returncode == 0 and "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-3000:]
        lines = r.stdout.splitlines()
        assert len(lines) == len(files)
        for f, line in zip(files, lines):
            res.append((line, open(f + ".out", "rb").read() if line.startswith("ok") else None))
    return res


def zlib_member(m):
    """what zlib makes of one member: its output when zlib inflates the deflate data to exactly the trailer and the output has the
    trailer's ISIZE and CRC-32, else None"""
    xlen = struct.unpack_from("<H", m, 10)[0]
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(m[12 + xlen:len(m) - 8])
    except zlib.error:
        return None
    crc, isize = struct.unpack("<II", m[-8:])
    if not d.eof or d.unused_data or len(out) != isize or zlib.crc32(out) != crc:
        return None
    return out


def inflate_zlib(blob):
    return b"".join(zlib_member(blob[o:o + n]) for o, n, _ in B.members(blob))


def test_host_decoder_matches_zlib(host):
    cases = B.cases()
    got = run_host(host, list(cases.values()))
    for (name, blob), (line, out) in zip(cases.items(), got):
        exp = inflate_zlib(blob)
        assert line == f"ok {len(exp)}", (name, line)
        assert out == exp, name


def small_members():
    text = B.pairs_text(40, 3)
    return {"dynamic": B.member(text[:1500]), "fixed": B.member(text[:400], strategy=zlib.Z_FIXED),
            "stored": B.member(text[:200], level=0), "blocks": B.member(text[:900], flush=zlib.Z_FULL_FLUSH, flush_every=250),
            "rle": B.member(b"ab" * 40 + b"\n" * 200 + text[:100], strategy=zlib.Z_RLE)}


def test_every_bit_flip_in_the_deflate_data_matches_zlib(host):
    """each flipped bit: an error exactly when zlib refuses the member (or its CRC / ISIZE no longer match), else zlib's bytes"""
    for name, m in small_members().items():
        d0 = 12 + struct.unpack_from("<H", m, 10)[0]
        blobs = []
        for bit in range(8 * d0, 8 * (len(m) - 8)):
            x = bytearray(m); x[bit >> 3] ^= 1 << (bit & 7); blobs.append(bytes(x))
        accepted = 0
        for x, (line, out) in zip(blobs, run_host(host, blobs)):
            exp = zlib_member(x)
            if exp is None:
                assert line.startswith("error: member 0 at byte 0: "), (name, line)
            else:
                accepted += 1
                assert line == f"ok {len(exp)}" and out == exp, (name, line)
        assert accepted < len(blobs) // 4, name                           # most flips are caught (padding bits are not)


def test_trailer_flips(host):
    m = small_members()["dynamic"]
    blobs = []
    for bit in range(64):
        x = bytearray(m); x[len(m) - 8 + (bit >> 3)] ^= 1 << (bit & 7); blobs.append(bytes(x))
    for bit, (line, out) in enumerate(run_host(host, blobs)):
        assert line.startswith("error: member 0 at byte 0: "), (bit, line)
        if bit < 32:
            assert line.endswith("CRC-32 mismatch"), line


def test_truncation_at_every_byte(host):
    """the file cut at every byte of a small member (the walk finds no whole member), and the member's deflate data cut at every
    byte with BSIZE rewritten to match (a whole member whose stream runs out)"""
    ms = small_members()
    m = ms["dynamic"]
    whole = B.member(b"x\n" * 100)
    blobs = [whole + m[:k] for k in range(1, len(m))]
    res = run_host(host, blobs)
    assert all(line == "error: member 1 at byte %d: truncated" % len(whole) for line, _ in res), res[:3]
    for name in ("dynamic", "fixed", "stored", "blocks"):
        m = ms[name]
        d0 = 12 + struct.unpack_from("<H", m, 10)[0]
        cut = []
        for k in range(d0, len(m) - 8):
            x = bytearray(m[:k] + m[-8:])
            struct.pack_into("<H", x, 16, len(x) - 1)                  # BSIZE: the BC subfield is the first one
            cut.append(bytes(x))
        for line, _ in run_host(host, cut):
            assert line.startswith("error: member 0 at byte 0: "), (name, line)


def test_header_refusals(host):
    m = small_members()["fixed"]
    past = bytearray(m); struct.pack_into("<H", past, 16, len(m) + 100)      # BSIZE past the end of the file
    big = bytearray(m); struct.pack_into("<I", big, len(m) - 4, 65537)        # ISIZE > 65536
    small = bytearray(m); struct.pack_into("<H", small, 16, 20)               # BSIZE below header + trailer
    res = run_host(host, [bytes(past), bytes(big), bytes(small), gzip.compress(b"a\tb\n"), b"plain text\n"])
    assert res[0][0] == "error: member 0 at byte 0: truncated"
    assert res[1][0] == "error: member 0 at byte 0: ISIZE larger than 64 KiB"
    assert res[2][0] == "error: member 0 at byte 0: BSIZE smaller than the header and trailer"
    assert "gzip but not BGZF" in res[3][0]
    assert res[4][0] == "error: member 0 at byte 0: not a gzip member"


# ---------------------------------------------------------------- mk_bgzf_scan (the library's host walk)
def test_scan_offsets_and_stop():
    blob = B.cases()["foreign_subfield"] + B.bgzf(B.pairs_text(3000, 5), level=1)
    exp = B.members(blob)
    mem, nb, n_out = mk.bgzf_scan(blob)
    assert [(m.in_off, m.in_len, m.isize) for m in mem] == exp
    assert [m.out_off for m in mem] == [sum(i for _, _, i in exp[:k]) for k in range(len(exp))]
    assert nb == len(blob) and n_out == sum(i for _, _, i in exp)
    for cut in (1, 17, exp[3][1] // 2, exp[3][1] - 1):                  # an incomplete fourth member: three whole ones
        mem, nb, n_out = mk.bgzf_scan(blob[:exp[3][0] + cut])
        assert len(mem) == 3 and nb == exp[3][0] and n_out == sum(i for _, _, i in exp[:3])
    mem, nb, _ = mk.bgzf_scan(blob, cap=2)                              # at most cap members
    assert len(mem) == 2 and nb == exp[2][0]
    assert mk.bgzf_scan(b"")[1:] == (0, 0)


def test_scan_refusals():
    with pytest.raises(mk.MkError, match="error -6: .*byte 0: gzip but not BGZF"):
        mk.bgzf_scan(gzip.compress(B.pairs_text(100)))
    good = B.member(b"a\n" * 50)
    with pytest.raises(mk.MkError, match=f"error -6: .*byte {len(good)}: not a gzip member"):
        mk.bgzf_scan(good + b"chr1\t5\n")
    big = bytearray(good); struct.pack_into("<I", big, len(good) - 4, 65537)
    with pytest.raises(mk.MkError, match=f"error -6: .*byte {len(good)}: ISIZE larger than 64 KiB"):
        mk.bgzf_scan(good + bytes(big))


def test_member_struct_mirror_matches_the_header(tmp_path):
    """mk_bgzf_member compiled by gcc has the size and field offsets of capi.BgzfMember"""
    import ctypes as C
    from microcket_b200 import capi
    f = capi.BgzfMember._fields_
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "microcket_b200.h"\nint main(void) { printf("%zu'
                   + " %zu" * len(f) + '\\n", sizeof(mk_bgzf_member)' + "".join(f", offsetof(mk_bgzf_member, {n})" for n, _ in f) + "); return 0; }\n")
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(tmp_path / "layout"), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(tmp_path / "layout")], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(capi.BgzfMember)] + [getattr(capi.BgzfMember, n).offset for n, _ in f]
