"""BGZF inflate on the GPU (csrc/bgzf.cu through capi.Bgzf and `pairs2bins x.pairs.gz`): byte-identical to Python's zlib on every
kind of member, the first damaged member named, refusals before any launch; and pairs2bins on bgzipped input byte-identical to
the run on the plain file, from a file and from stdin, across chunk boundaries and concatenated files."""
import os
import struct
import subprocess
import zlib

import pytest

import microcket_b200 as mk
import bgzf_corpus as B
from test_bgzf import inflate_zlib, small_members, zlib_member
from test_gpu_norm import BIN, NAMES, toy_pairs
from test_gpu_pairs import HG38_LEN

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def dev(blob, pad=0):
    t = torch.zeros(len(blob) + pad + 1, dtype=torch.uint8, device="cuda")
    if blob:
        t[pad:pad + len(blob)] = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    return t


def inflate(bz, blob, pad=0, out_cap=None):
    mem, nb, n_out = mk.bgzf_scan(blob)
    assert nb == len(blob)
    d_in = dev(blob, pad)
    out = torch.full((max(n_out, 1) + 64,), 0xA5, dtype=torch.uint8, device="cuda")
    bz.inflate(d_in.data_ptr() + pad, mem, out.data_ptr(), n_out if out_cap is None else out_cap)
    torch.cuda.synchronize()
    return out[:n_out].cpu().numpy().tobytes(), out


# ---------------------------------------------------------------- library
def test_matches_zlib_on_the_corpus():
    bz = mk.Bgzf(4096)
    for name, blob in B.cases(1).items():
        got, _ = inflate(bz, blob)
        assert got == inflate_zlib(blob), name
    assert mk.bgzf_decompress(B.bgzf(b"")) == b""
    bz.close()


def test_20000_members_in_one_call_two_calls_and_another_allocation():
    text = B.pairs_text(420000, 7)
    blob = B.bgzf(text, block=len(text) // 20500, level=1) + B.bgzf(text[:3000000], block=B.BLOCK, strategy=zlib.Z_RLE)
    mem, _, n_out = mk.bgzf_scan(blob)
    assert len(mem) > 20000
    exp = text + text[:3000000]
    bz = mk.Bgzf(len(mem))
    a, _ = inflate(bz, blob)
    b, _ = inflate(bz, blob)
    c, _ = inflate(bz, blob, pad=13)                                    # the same bytes at an odd offset of another tensor
    assert a == exp and b == exp and c == exp
    nl, last = bz.text_stats()
    assert nl == exp.count(b"\n") and last == exp.rfind(b"\n")
    bz.close()


def test_damaged_members_name_the_first_bad_one():
    """the members the host test proved safe, each between two good ones: an error exactly where zlib refuses, naming member 1"""
    good = B.member(B.pairs_text(300, 2)[:8000])
    bz = mk.Bgzf(8)
    for name, m in small_members().items():
        d0 = 12 + struct.unpack_from("<H", m, 10)[0]
        for bit in list(range(8 * d0, 8 * len(m), 3 if name == "dynamic" else 1)):
            x = bytearray(m); x[bit >> 3] ^= 1 << (bit & 7); x = bytes(x)
            if B.members(x)[0][2] > 65536:
                continue                                                # the walk refuses an ISIZE above 64 KiB
            exp = zlib_member(x)
            if exp is None:
                with pytest.raises(mk.MkError, match="error -6: BGZF member 1 "):
                    inflate(bz, good + x + good)
            else:
                assert inflate(bz, good + x + good)[0] == zlib_member(good) + exp + zlib_member(good)
    bad = bytearray(good); bad[40] ^= 0xFF
    with pytest.raises(mk.MkError, match="BGZF member 2 "):                  # the first of two damaged members, in file order
        inflate(bz, good + good + bytes(bad) + good + bytes(bad))
    bz.close()


def test_out_cap_one_byte_short_is_refused_before_any_launch():
    blob = B.bgzf(B.pairs_text(2000, 4))
    mem, _, n_out = mk.bgzf_scan(blob)
    bz = mk.Bgzf(len(mem))
    launches = bz.launches()
    with pytest.raises(mk.MkError, match="error -1"):
        inflate(bz, blob, out_cap=n_out - 1)
    assert bz.launches() == launches
    d_in, out = dev(blob), torch.empty(n_out, dtype=torch.uint8, device="cuda")
    with pytest.raises(mk.MkError, match="error -4"):                   # more members than the object holds
        mk.Bgzf(1).inflate(d_in.data_ptr(), mem, out.data_ptr(), n_out)
    bz.close()


# ---------------------------------------------------------------- pairs2bins
def run(cmd, **kw):
    return subprocess.run(cmd, capture_output=True, **kw)


@pytest.fixture(scope="module")
def pairs(tmp_path_factory):
    d = tmp_path_factory.mktemp("bgzf_cli")
    p = toy_pairs(HG38_LEN, 60000, 17)
    lines = [f"r{i}\t{NAMES[a]}\t{x}\t{NAMES[b]}\t{y}\t+\t-\n" for i, (a, x, b, y) in
             enumerate(zip(p["chr1"].tolist(), p["pos1"].tolist(), p["chr2"].tolist(), p["pos2"].tolist()))]
    text = ("## pairs format v1.0\n#sorted: none\n#columns: readID chr1 pos1 chr2 pos2 strand1 strand2\n"
            + "".join(lines + lines[:3000])).encode()[:-1]                  # duplicates, and no final newline
    (d / "x.pairs").write_bytes(text)
    (d / "hg38.info").write_text("".join(f"{n}\t{l}\n" for n, l in zip(NAMES, HG38_LEN)))
    return d, text


def outputs(d, prefix, res, hic):
    got = {f"{r}.{ext}": (d / f"{prefix}.{r}.{ext}").read_bytes() for r in res for ext in ("coo", "bins.bed") if (d / f"{prefix}.{r}.{ext}").exists()}
    if hic:
        got["hic"] = (d / f"{prefix}.hic").read_bytes()
    return got


def same_as_plain(d, gz_bytes, args, res, hic=False, stdin=False, env=None):
    exe = os.path.join(BIN, "pairs2bins")
    (d / "x.pairs.gz").write_bytes(gz_bytes)
    e = {**os.environ, **(env or {})}
    out = {}
    for tag, src in (("p", "x.pairs"), ("g", "x.pairs.gz")):
        h = ["-H", str(d / f"{tag}.hic")] if hic else []
        if stdin and tag == "g":
            r = run([exe] + h + args + ["-", str(d / tag), str(d / "hg38.info")], input=gz_bytes, env=e)
        else:
            r = run([exe] + h + args + [str(d / src), str(d / tag), str(d / "hg38.info")], env=e)
        assert r.returncode == 0, r.stderr
        out[tag] = (r.stderr, outputs(d, tag, res, hic))
    assert out["g"][1] and out["g"] == out["p"]
    return out["p"][0].decode()


def test_cli_dense_sort_and_hic_with_norms(pairs):
    d, text = pairs
    res = [1000000, 100000, 50000]
    err = same_as_plain(d, B.bgzf(text), ["-b", "-n", "VC,KR,GW_KR", "-r", ",".join(map(str, res))], res, hic=True,
                        env={"MICROCKET_DENSE_MB": "64"})
    lines = text.count(b"\n") + 1                                       # the last line has no newline
    assert f"INFO: {lines} lines" in err and "INFO: GW_KR at 100000 bp" in err


def test_cli_dedup_from_stdin_in_1_mib_chunks(pairs):
    d, text = pairs
    res = [1000000, 5000]
    gz = B.bgzf(text, block=30000, level=9, strategy=zlib.Z_FILTERED)
    assert len(text) > 2 << 20
    err = same_as_plain(d, gz, ["-d", "-r", ",".join(map(str, res))], res, stdin=True, env={"MICROCKET_CHUNK_MB": "1"})
    assert "after duplicate removal" in err


def test_cli_concatenated_files_with_eof_members(pairs):
    d, text = pairs
    k = len(text) // 3 + 7                                               # inside a line
    gz = B.bgzf(text[:k], level=1) + B.EOF + B.bgzf(text[k:], block=B.BLOCK - 1, level=6)
    same_as_plain(d, gz, ["-r", "1000000,100000"], [1000000, 100000], env={"MICROCKET_CHUNK_MB": "1"})


def test_cli_refusals(pairs):
    import gzip
    d, text = pairs
    exe = os.path.join(BIN, "pairs2bins")
    args = ["-r", "1000000", str(d / "y.pairs.gz"), str(d / "o"), str(d / "hg38.info")]
    (d / "y.pairs.gz").write_bytes(gzip.compress(text[:100000]))
    r = run([exe] + args)
    assert r.returncode == 10 and b"gzip but not BGZF" in r.stderr and b"zcat" in r.stderr, r.stderr
    gz = B.bgzf(text[:400000])
    (d / "y.pairs.gz").write_bytes(gz[:len(gz) - 28 - 100])             # the last data member cut short
    r = run([exe] + args)
    assert r.returncode == 10 and b"truncated" in r.stderr, r.stderr
    bad = bytearray(gz); bad[B.members(gz)[3][0] + 30] ^= 0x10
    (d / "y.pairs.gz").write_bytes(bytes(bad))
    r = run([exe] + args)
    assert r.returncode == 10 and b"Error: " in r.stderr and b"BGZF member 3 " in r.stderr, r.stderr
