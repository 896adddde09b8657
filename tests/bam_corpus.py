"""SAM lines for the BAM encoder's tests (tests/test_bam_encode.py on the host form, tests/test_gpu_sam2bam.py on the device and
the `sam2bam` executable): every field and tag type, and one line per refusal with the code bam_encode.h gives it."""
import struct

import numpy as np

REFS = [("chr1", 248956422), ("chr2", 242193529), ("chrM", 16569), ("scaffold_7", 40000)]

_REC = [
    # plain mapped pairs, '=' and explicit RNEXT, '*' fields
    "r1\t99\tchr1\t100\t60\t10M\t=\t300\t210\tACGTACGTAC\tIIIIIIIIII",
    "r1\t147\tchr1\t300\t60\t10M\t=\t100\t-210\tACGTACGTAC\tIIIIIIIIII",
    "r2\t65\tchr1\t16380\t30\t5M2I3M\tchr2\t5000\t0\tacgtnNRYKM\t!!!!!!!!!!",
    "r3\t0\tchr2\t1\t255\t*\t*\t0\t0\t*\t*",
    "r4\t16\tchrM\t16000\t0\t3S5M1D2M3H\t*\t0\t0\tAC=MGRSVTW\t*",
    "r5\t0\tscaffold_7\t32760\t7\t20M\t*\t0\t0\tACGTACGTACGTACGTACGTA\t*",                         # odd l_seq (21)
    "r6\t4\t*\t0\t0\t*\t*\t0\t0\tACG\tIII",                                                      # unmapped, no coordinate
    "r7\t4\tchr1\t5000\t0\t*\tchr1\t5000\t0\tACGT\tIIII",                                          # placed unmapped, no CIGAR
    "r8\t4\tchr1\t16383\t0\t50M\t=\t16383\t0\tACGT\tIIII",                                         # placed unmapped with CIGAR
    "r9\t0\tchr1\t1000\t60\t4M1000N4M2P1=1X\t*\t0\t0\tACGTACGTAC\tJJJJJJJJJJ",
    # integer tags at every type boundary
    "t1\t0\tchr2\t10\t1\t1M\t*\t0\t0\tA\tI\tX0:i:-129\tX1:i:-128\tX2:i:255\tX3:i:256\tX4:i:65535\tX5:i:65536\tX6:i:4294967295",
    "t2\t0\tchr2\t10\t1\t1M\t*\t0\t0\tA\tI\tY0:i:-32768\tY1:i:-32769\tY2:i:-2147483648\tY3:i:0\tY4:i:127\tY5:i:-1",
    "t3\t0\tchr2\t11\t1\t1M\t*\t0\t0\tA\tI\tAA:A:x\tZZ:Z:hello world\tZE:Z:\tHH:H:1AE301",
    # B arrays, all seven subtypes, empty arrays
    "t4\t0\tchr2\t12\t1\t1M\t*\t0\t0\tA\tI\tBc:B:c,-128,0,127\tBC:B:C,0,255\tBs:B:s,-32768,32767\tBS:B:S,0,65535",
    "t5\t0\tchr2\t12\t1\t1M\t*\t0\t0\tA\tI\tBi:B:i,-2147483648,2147483647\tBI:B:I,0,4294967295\tBf:B:f,1.5,-0.25,3\tBe:B:c",
    # floats on the fast path and off it
    "f1\t0\tchr2\t13\t1\t1M\t*\t0\t0\tA\tI\tF0:f:1.5\tF1:f:-0.1\tF2:f:3e10\tF3:f:16777216\tF4:f:0.0000000001\tF5:f:-0",
    "f2\t0\tchr2\t13\t1\t1M\t*\t0\t0\tA\tI\tG0:f:0.1234567891\tG1:f:1e-20\tG2:f:3.4e38\tG3:f:16777217\tG4:f:1e11\tG5:f:123456789012345678901234",
    "f3\t0\tchr2\t14\t1\t1M\t*\t0\t0\tA\tI\tBf:B:f,0.333333333333,2.5e-12,7",
    "f4\t0\tchr2\t14\t1\t1M\t*\t0\t0\tA\tI\tF0:f:.5\tF1:f:5.\tF2:f:+2.25E+3\tF3:f:1E-10",
    # a long QNAME (254), many CIGAR ops
    "q" * 254 + "\t0\tchr1\t7\t1\t" + "1M1I" * 300 + "\t*\t0\t0\t" + "A" * 600 + "\t*",
]

CORPUS = "\n".join(_REC) + "\n"

# one refused line each, with bam_encode.h's code (BE_E*)
REFUSALS = [
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*", 1),                              # 10 fields
    ("q" * 255 + "\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*", 2),
    ("a\t0x10\tchr1\t1\t0\t*\t*\t0\t0\t*\t*", 3),
    ("a\t65536\tchr1\t1\t0\t*\t*\t0\t0\t*\t*", 3),
    ("a\t0\tchr9\t1\t0\t*\t*\t0\t0\t*\t*", 4),
    ("a\t0\tchr1\t-1\t0\t*\t*\t0\t0\t*\t*", 5),
    ("a\t0\tchr1\t2147483648\t0\t*\t*\t0\t0\t*\t*", 5),
    ("a\t0\tchr1\t1\t256\t*\t*\t0\t0\t*\t*", 6),
    ("a\t0\tchr1\t1\t0\t10Q\t*\t0\t0\t*\t*", 7),
    ("a\t0\tchr1\t1\t0\tM\t*\t0\t0\t*\t*", 7),
    ("a\t0\tchr1\t1\t0\t10M5\t*\t0\t0\t*\t*", 7),
    ("a\t0\tchr1\t1\t0\t" + "1M" * 65536 + "\t*\t0\t0\t*\t*", 8),
    ("a\t0\tchr1\t1\t0\t*\tchrX\t0\t0\t*\t*", 9),
    ("a\t0\tchr1\t1\t0\t*\t*\tx\t0\t*\t*", 10),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t2147483648\t*\t*", 11),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\tACGT\tIII", 12),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\tIII", 12),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXXi:1", 13),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXX:i:", 13),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXX:Q:1", 14),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXX:B:q,1", 15),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXX:i:4294967296", 16),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXX:i:-2147483649", 16),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXX:B:C,256", 16),
    ("a\t0\tchr1\t1\t0\t*\t*\t0\t0\t*\t*\tXX:f:1.2.3", 17),
    ("a\t0\tchr1\t0\t0\t*\t*\t0\t0\t*\t*", 18),
    ("@CO\tlate header", 19),
]


def expected_records(text, refs=REFS):
    """encode_records of the text, with the bin of flag-4 records that have a CIGAR set to reg2bin(pos, pos + 1)"""
    import bam_writer
    out = bytearray(bam_writer.encode_records(text, refs))
    p = 0
    while p < len(out):
        n = struct.unpack_from("<I", out, p)[0]
        pos, flag = struct.unpack_from("<i", out, p + 8)[0], struct.unpack_from("<H", out, p + 18)[0]
        if flag & 4 and pos >= 0:
            struct.pack_into("<H", out, p + 14, bam_writer._reg2bin(pos, pos + 1))
        p += 4 + n
    return bytes(out)


def split_records(blob):
    out, p = [], 0
    while p < len(blob):
        n = struct.unpack_from("<I", blob, p)[0]
        out.append(blob[p:p + 4 + n]); p += 4 + n
    return out


def sort_key(rec, n_ref):
    tid, pos = struct.unpack_from("<ii", rec, 4)
    flag = struct.unpack_from("<H", rec, 18)[0]
    return (n_ref if tid < 0 else tid, pos + 1, flag >> 4 & 1)


def sorted_records(blob, n_ref):
    """the records in the stable (tid', pos + 1, rev) order, by numpy's lexsort"""
    recs = split_records(blob)
    if not recs:
        return []
    k = np.array([sort_key(r, n_ref) for r in recs], dtype=np.int64)
    order = np.lexsort((k[:, 2], k[:, 1], k[:, 0]))
    return [recs[i] for i in order]


def header(refs=REFS, hd="@HD\tVN:1.6\tSO:unsorted"):
    lines = ([hd] if hd else []) + [f"@SQ\tSN:{n}\tLN:{l}" for n, l in refs]
    return "\n".join(lines) + "\n"
