"""SAM -> BAM records without a GPU: the host form of the per-line encoder (csrc/bam_encode.h, the code every thread of
bam_out.cu runs on one line, through tests/bam_encode_host.cpp) built with AddressSanitizer and UBSan.  Its bytes must equal
tests/bam_writer.encode_records (an encoder written from SAMv1) on a corpus covering every field and tag type, and every
refusal must name the right line.  The usage refusals of `sam2bam`, which come before any device call, are checked too."""
import os
import shutil
import subprocess

import pytest

import microcket_b200 as mk
import bam_corpus as BC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAM2BAM = os.path.join(os.path.dirname(mk.LIB_PATH), "bin", "sam2bam")


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("bam_encode_host")
    exe = str(d / "bam_encode_host")
    subprocess.run([cxx, "-std=c++17", "-g", "-O1", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                    "-I", os.path.join(ROOT, "microcket_b200", "csrc"), os.path.join(ROOT, "tests", "bam_encode_host.cpp"), "-o", exe],
                   check=True)
    refs = d / "refs.txt"
    refs.write_text("".join(f"{n}\t{l}\n" for n, l in BC.REFS))

    def run(text):
        (d / "in.sam").write_bytes(text.encode())
        r = subprocess.run([exe, str(refs), str(d / "in.sam"), str(d / "out.bin")], capture_output=True, text=True,
                           env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
        assert "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr
        return r.returncode, (d / "out.bin").read_bytes() if r.returncode == 0 else b"", r.stderr
    return run


def test_corpus_bytes_equal_bam_writer(host):
    rc, got, err = host(BC.CORPUS)
    assert rc == 0, err
    exp = BC.expected_records(BC.CORPUS)
    assert len(BC.split_records(got)) == len(BC.CORPUS.splitlines())
    for k, (a, b) in enumerate(zip(BC.split_records(got), BC.split_records(exp))):
        assert a == b, f"record {k}: {BC.CORPUS.splitlines()[k][:80]}"
    assert got == exp


def test_unmapped_with_cigar_gets_one_base_bin(host):
    """the one deliberate difference from encode_records: flag 4 + CIGAR -> bin of [pos, pos + 1)"""
    import bam_writer
    line = "u\t4\tchr1\t16380\t0\t50M\t*\t0\t0\tACGT\tIIII\n"          # 50M from 16379 would cross the 16 kb boundary
    rc, got, _ = host(line)
    ref = bam_writer.encode_records(line, BC.REFS)
    assert rc == 0 and int.from_bytes(got[14:16], "little") == 4681 and int.from_bytes(ref[14:16], "little") == 585
    assert got[:14] + got[16:] == ref[:14] + ref[16:]


@pytest.mark.parametrize("k", range(len(BC.REFUSALS)))
def test_refusal_names_the_line(host, k):
    bad, code = BC.REFUSALS[k]
    good = BC.CORPUS.splitlines()
    at = (7 * k) % (len(good) + 1)
    lines = good[:at] + [bad] + good[at:] + [BC.REFUSALS[(k + 1) % len(BC.REFUSALS)][0]]   # a later bad line does not win
    rc, _, err = host("\n".join(lines) + "\n")
    assert rc == 10
    assert err.startswith(f"line {at + 1} code {code}:"), err


def test_sam2bam_usage():
    if not os.path.exists(SAM2BAM):
        pytest.skip("bin/sam2bam is not built")
    for args in ([], ["-x"], ["-o"], ["in.sam"], ["-o", "a.bam", "-o", "b.bam"]):
        r = subprocess.run([SAM2BAM] + args, capture_output=True, text=True)
        assert r.returncode == 2 and "Usage" in r.stderr, args
    r = subprocess.run([SAM2BAM, "-h"], capture_output=True, text=True)
    assert r.returncode == 0 and "MICROCKET_SORT_MB" in r.stderr
