"""BGZF deflate members written as one fixed-Huffman block (RFC 1951 §3.2.6) that hold literals 144-255, which take the 9-bit
fixed codes.  Small members of binary data (a BAM header, the short last member of a BAM record stream) choose the fixed block;
.pairs text never has such bytes.  zlib must inflate every member to its input: on the host form of the encoder
(csrc/bgzf_deflate.h, built with AddressSanitizer and UBSan) and on the device, whose bytes must equal the host form's."""
import os
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest

import microcket_b200 as mk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def inputs():
    """small inputs over few byte values (so that a fixed block wins) with literals on both sides of 144, and a BAM header"""
    rng = np.random.default_rng(5)
    out = []
    for n in (16, 40, 100, 193, 300, 700):
        for alpha in ((0, 0xc6, 0xd6, 0x0e), (0x90, 0xff, 0x41), tuple(range(140, 150))):
            out.append(bytes(rng.choice(alpha, n).astype(np.uint8)))
    text = "@HD\tVN:1.4\tSO:coordinate\n@SQ\tSN:chr1\tLN:248956422\n@SQ\tSN:chrM\tLN:16569\n"
    hdr = b"BAM\1" + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", 2)
    for name, ln in (("chr1", 248956422), ("chrM", 16569)):
        hdr += struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", ln)
    out.append(hdr)
    return out


def members(blob):
    p, out = 0, []
    while p < len(blob):
        bs = struct.unpack_from("<H", blob, p + 16)[0] + 1
        out.append(blob[p:p + bs]); p += bs
    return out


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("bgzf_fixed")
    exe = str(d / "bgzf_deflate_host")
    subprocess.run([cxx, "-std=c++17", "-g", "-O1", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                    "-I", os.path.join(ROOT, "microcket_b200", "csrc"), os.path.join(ROOT, "tests", "bgzf_deflate_host.cpp"), "-o", exe],
                   check=True)

    def run(data):
        (d / "in").write_bytes(data)
        r = subprocess.run([exe, "c", "-1", str(d / "in"), str(d / "out")], capture_output=True, text=True,
                           env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
        assert r.returncode == 0 and "runtime error" not in r.stderr, r.stderr
        return (d / "out").read_bytes()
    return run


def test_fixed_blocks_with_high_literals_inflate(host):
    fixed_high = 0
    for data in inputs():
        (m,) = members(host(data))
        assert zlib.decompress(m[18:-8], -15) == data
        assert struct.unpack("<I", m[-8:-4])[0] == zlib.crc32(data)
        fixed_high += (m[18] & 7) == 3 and max(data) >= 144        # BFINAL + BTYPE 01
    assert fixed_high >= 3


@pytest.mark.gpu
def test_device_fixed_blocks_equal_host(host):
    pytest.importorskip("torch")
    for data in inputs():
        dev = mk.bgzf_compress(data, eof=False)
        assert dev == host(data)
        assert zlib.decompress(dev[18:-8], -15) == data
