"""BGZF deflate on the GPU (csrc/bgzf_deflate.cu through capi.BgzfDeflate and `bgzip`): every output read back by gzip, by raw zlib
member by member and by the project's inflate; byte-identical to the host form (tests/bgzf_deflate_host.cpp) and deterministic
across calls, addresses, streams and call cuts; refusals before any launch; and the drop-in CLI."""
import gzip
import os
import subprocess
import zlib

import pytest

import microcket_b200 as mk
import bgzf_corpus as B
from test_bgzf_deflate import BGZIP, check_members, host, host_compress, inputs, sorted_text  # noqa: F401  (host: a fixture)
from test_gpu_bgzf import pairs  # noqa: F401  (a fixture)
from test_gpu_bgzf import same_as_plain

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def dev(data, pad=0):
    t = torch.zeros(len(data) + pad + 1, dtype=torch.uint8, device="cuda")
    if data:
        t[pad:pad + len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    return t


def deflate(bd, data, level=-1, pad=0, stream=0):
    d_in = dev(data, pad)
    cap = mk.bgzf_deflate_bound(len(data))
    out = torch.full((cap + 64,), 0xA5, dtype=torch.uint8, device="cuda")
    n, mem = bd.deflate(d_in.data_ptr() + pad, len(data), out.data_ptr(), cap, level, stream)
    torch.cuda.synchronize()
    return out[:n].cpu().numpy().tobytes(), mem


def table(mem):
    return [(m.in_off, m.in_len, m.out_off, m.isize) for m in mem]


def check(blob, mem, data, bz):
    check_members(blob, data)
    scan, nb, n_out = mk.bgzf_scan(blob)
    assert nb == len(blob) and n_out == len(data) and table(mem) == table(scan)
    if data:
        d_in, out = dev(blob), torch.empty(len(data) + 1, dtype=torch.uint8, device="cuda")
        bz.inflate(d_in.data_ptr(), scan, out.data_ptr(), len(data))
        torch.cuda.synchronize()
        assert out[:len(data)].cpu().numpy().tobytes() == data


def test_round_trips_and_equals_the_host_form(host):
    bd, bz = mk.BgzfDeflate(4 << 20), mk.Bgzf(4096)
    for name, data in inputs(1).items():
        blob, mem = deflate(bd, data)
        check(blob, mem, data, bz)
        assert blob == host_compress(host, data), name
        assert deflate(bd, data, level=1)[0] == blob and deflate(bd, data, level=9)[0] == blob, name
        stored, smem = deflate(bd, data, level=0)
        check(stored, smem, data, bz)
        assert all(m.in_len == m.isize + 31 for m in smem) and stored == host_compress(host, data, 0), name
        if name == "random":
            assert blob == stored
    assert mk.bgzf_compress(b"") == B.EOF and gzip.decompress(mk.bgzf_compress(b"x\n" * 9)) == b"x\n" * 9
    bd.close(); bz.close()


def test_no_larger_than_zlib_level_1():
    text = B.pairs_text(300_000, seed=3)
    for data in (text, sorted_text(text)):
        z1 = sum(len(B.member(data[p:p + B.BLOCK], level=1)) for p in range(0, len(data), B.BLOCK))
        got = mk.bgzf_compress(data, eof=False)
        assert gzip.decompress(got + B.EOF) == data and len(got) <= z1


def test_deterministic_across_calls_addresses_streams_cuts_and_reuse():
    text = B.pairs_text(420000, 7)
    bd, bz = mk.BgzfDeflate(len(text)), mk.Bgzf(64)
    a, mem = deflate(bd, text)
    assert len(mem) > 250
    assert deflate(bd, text)[0] == a
    assert deflate(bd, text, pad=13)[0] == a                              # the same bytes at an odd address
    s = torch.cuda.Stream()
    assert deflate(bd, text, stream=s.cuda_stream)[0] == a
    cut = 7 * B.BLOCK                                                   # two calls cut at a multiple of 65 280
    assert deflate(bd, text[:cut])[0] + deflate(bd, text[cut:])[0] == a
    check(*deflate(bd, text[:200000]), text[:200000], bz)               # an inflate between two calls on the same objects
    assert deflate(bd, text)[0] == a
    bd.close(); bz.close()


def test_more_than_20000_members_in_one_call():
    """1.3 GB of input made and checked on the device; the host holds the compressed bytes and a sample of members only"""
    n = 20100 * B.BLOCK + 777
    unit = torch.frombuffer(bytearray(B.pairs_text(60000, 9)), dtype=torch.uint8).cuda()
    d_in = unit.repeat(-(-n // unit.numel()))[:n].contiguous()
    cap = mk.bgzf_deflate_bound(n)
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    bd = mk.BgzfDeflate(n)
    k, mem = bd.deflate(d_in.data_ptr(), n, out.data_ptr(), cap)
    bd.close()
    assert len(mem) == 20101
    blob = out[:k].cpu().numpy().tobytes()
    scan, nb, n_out = mk.bgzf_scan(blob, cap=len(mem) + 1)
    assert nb == k and n_out == n and table(mem) == table(scan)
    for i in list(range(0, len(mem), 997)) + [len(mem) - 1]:             # sampled members, each alone through raw zlib
        m = mem[i]
        assert blob[m.in_off:m.in_off + 16] == bytes.fromhex("1f8b08040000000000ff060042430200")
        got = zlib.decompress(blob[m.in_off + 18:m.in_off + m.in_len - 8], -15)
        assert got == d_in[m.out_off:m.out_off + m.isize].cpu().numpy().tobytes()
    del blob
    bz = mk.Bgzf(len(scan))
    back = torch.empty(n, dtype=torch.uint8, device="cuda")
    bz.inflate(out.data_ptr(), scan, back.data_ptr(), n)                # every member, its CRC-32 and ISIZE checked on the device
    torch.cuda.synchronize()
    bz.close()
    assert torch.equal(back, d_in)
    del back
    bd = mk.BgzfDeflate(n)                                              # another object, another allocation: the same bytes
    out2 = torch.empty(cap, dtype=torch.uint8, device="cuda")
    k2, _ = bd.deflate(d_in.data_ptr(), n, out2.data_ptr(), cap)
    bd.close()
    torch.cuda.synchronize()
    assert k2 == k and torch.equal(out2[:k], out[:k])


def test_refusals_before_any_launch():
    data = B.pairs_text(3000, 2)
    bd = mk.BgzfDeflate(len(data))
    d_in = dev(data)
    cap = mk.bgzf_deflate_bound(len(data))
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    L = mk.lib()
    import ctypes as C
    n_out, nm = C.c_size_t(), C.c_size_t()
    mem = (mk.BgzfMember * 8)()
    launches = bd.launches()
    cases = [(bd.h, d_in.data_ptr(), len(data), -1, out.data_ptr(), cap - 1, C.byref(n_out), mem, 8, C.byref(nm), None),      # out_cap
             (bd.h, d_in.data_ptr(), len(data) + 1, -1, out.data_ptr(), cap + 99, C.byref(n_out), mem, 8, C.byref(nm), None),  # n > max_bytes
             (bd.h, d_in.data_ptr(), len(data), 10, out.data_ptr(), cap, C.byref(n_out), mem, 8, C.byref(nm), None),          # level
             (bd.h, d_in.data_ptr(), len(data), -2, out.data_ptr(), cap, C.byref(n_out), mem, 8, C.byref(nm), None),
             (bd.h, None, len(data), -1, out.data_ptr(), cap, C.byref(n_out), mem, 8, C.byref(nm), None),                     # null pointers
             (bd.h, d_in.data_ptr(), len(data), -1, None, cap, C.byref(n_out), mem, 8, C.byref(nm), None),
             (bd.h, d_in.data_ptr(), len(data), -1, out.data_ptr(), cap, None, mem, 8, C.byref(nm), None),
             (None, d_in.data_ptr(), len(data), -1, out.data_ptr(), cap, C.byref(n_out), mem, 8, C.byref(nm), None),
             (bd.h, d_in.data_ptr(), len(data), -1, out.data_ptr(), cap, C.byref(n_out), mem, 0, C.byref(nm), None)]          # table too small
    for k, args in enumerate(cases):
        assert L.L.mk_bgzf_deflate_device(*args) in (-1, -4), k
    assert bd.launches() == launches
    assert L.L.mk_bgzf_deflate_device(*cases[0][:5], cap, *cases[0][6:]) == 0 and bd.launches() == launches + 3
    bd.close()


# ---------------------------------------------------------------- bgzip
def run(cmd, **kw):
    return subprocess.run(cmd, capture_output=True, **kw)


def test_cli_file_keep_stdout_stdin_force_and_decompress(tmp_path):
    text = B.pairs_text(150000, 4)
    exp = mk.bgzf_compress(text)
    f = tmp_path / "x.pairs"
    f.write_bytes(text)
    r = run([BGZIP, "-@", "8", str(f)])
    assert r.returncode == 0, r.stderr
    assert not f.exists() and (tmp_path / "x.pairs.gz").read_bytes() == exp and gzip.decompress(exp) == text
    f.write_bytes(text)
    r = run([BGZIP, "-k", str(f)])                                      # the output exists: refused without -f
    assert r.returncode == 10 and b"-f" in r.stderr and f.exists()
    (tmp_path / "x.pairs.gz").write_bytes(b"old")
    r = run([BGZIP, "-kf", "-l", "6", str(f)])
    assert r.returncode == 0 and f.read_bytes() == text and (tmp_path / "x.pairs.gz").read_bytes() == exp
    assert run([BGZIP, "-c", str(f)]).stdout == exp and f.exists()
    assert run([BGZIP], input=text).stdout == exp and run([BGZIP, "-"], input=text).stdout == exp
    assert run([BGZIP, "-l0", "-c", str(f)]).stdout == mk.bgzf_compress(text, level=0)
    r = run([BGZIP, "-c", str(f)], env={**os.environ, "MICROCKET_CHUNK_MB": "1"})
    assert r.returncode == 0 and r.stdout == exp                        # 1 MiB chunks: the same bytes
    os.remove(f)
    r = run([BGZIP, "-d", str(tmp_path / "x.pairs.gz")])
    assert r.returncode == 0 and f.read_bytes() == text and not (tmp_path / "x.pairs.gz").exists()
    assert run([BGZIP, "-d"], input=exp).stdout == text
    assert run([BGZIP, "-dc", "-"], input=B.bgzf(text, level=9)).stdout == text   # zlib's BGZF too
    (tmp_path / "y.gz").write_bytes(gzip.compress(text))
    r = run([BGZIP, "-d", str(tmp_path / "y.gz")])
    assert r.returncode == 10 and b"not BGZF" in r.stderr and not (tmp_path / "y").exists() and (tmp_path / "y.gz").exists()
    e = tmp_path / "e"
    e.write_bytes(b"")
    assert run([BGZIP, str(e)]).returncode == 0 and (tmp_path / "e.gz").read_bytes() == B.EOF and not e.exists()
    assert run([BGZIP, "-d", str(tmp_path / "e.gz")]).returncode == 0 and e.read_bytes() == b""


def test_cli_pairs_gz_feeds_pairs2bins(pairs):  # noqa: F811
    d, text = pairs
    (d / "c.pairs").write_bytes(text)
    r = run([BGZIP, "-f", str(d / "c.pairs")])
    assert r.returncode == 0, r.stderr
    res = [1000000, 100000]
    same_as_plain(d, (d / "c.pairs.gz").read_bytes(), ["-r", ",".join(map(str, res))], res, hic=True)
