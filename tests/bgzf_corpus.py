"""BGZF writer with zlib's level / strategy / flush options, and the inputs the inflate tests run on (tests/test_bgzf.py on the
CPU, tests/test_gpu_bgzf.py on the GPU).  Written from SAMv1 §4.1 and RFC 1952; the only compressor is Python's zlib."""
import struct
import zlib

import numpy as np

BLOCK = 65280                                                          # bgzip's member payload
EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def member(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush=None, flush_every=0, foreign=b""):
    """one BGZF member holding `data` (<= 64 KiB); flush / flush_every: zlib.Z_SYNC_FLUSH or Z_FULL_FLUSH every so many bytes
    (several blocks, empty stored blocks); foreign: extra subfields written ahead of BC"""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    if flush and flush_every:
        cd = b"".join(c.compress(data[i:i + flush_every]) + c.flush(flush) for i in range(0, len(data), flush_every))
    else:
        cd = c.compress(data)
    cd += c.flush()
    extra = foreign + b"BC" + struct.pack("<H", 2)
    total = 12 + len(extra) + 2 + len(cd) + 8
    assert total <= 65536, total
    extra += struct.pack("<H", total - 1)
    return b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", len(extra)) + extra + cd + struct.pack("<II", zlib.crc32(data), len(data))


def bgzf(data, block=BLOCK, eof=True, **kw):
    """`data` in members of `block` bytes (the last one shorter), then the EOF member"""
    out = [member(data[p:p + block], **kw) for p in range(0, len(data), block)]
    return b"".join(out) + (EOF if eof else b"")


def members(blob):
    """[(offset, length, isize)] of a well-formed BGZF byte string (an independent walk for the tests)"""
    out, p = [], 0
    while p < len(blob):
        xlen = struct.unpack_from("<H", blob, p + 10)[0]
        x, bsize = 0, None
        while x + 4 <= xlen:
            si1, si2, sl = blob[p + 12 + x], blob[p + 13 + x], struct.unpack_from("<H", blob, p + 14 + x)[0]
            if (si1, si2, sl) == (66, 67, 2):
                bsize = struct.unpack_from("<H", blob, p + 16 + x)[0]
            x += 4 + sl
        n = bsize + 1
        out.append((p, n, struct.unpack_from("<I", blob, p + n - 4)[0]))
        p += n
    return out


def pairs_text(n, seed=0):
    """4DN-style .pairs lines (header included), the kind of text the members of a .pairs.gz hold"""
    rng = np.random.default_rng(seed)
    names = [f"chr{i}" for i in range(1, 23)] + ["chrX", "chrY"]
    c1, c2 = rng.integers(0, len(names), n), rng.integers(0, len(names), n)
    p1, p2 = rng.integers(1, 150_000_000, n), rng.integers(1, 150_000_000, n)
    s = rng.integers(0, 4, n)
    lines = ["## pairs format v1.0\n#columns: readID chr1 pos1 chr2 pos2 strand1 strand2\n"]
    lines += [f"SRR{seed}.{i}\t{names[a]}\t{x}\t{names[b]}\t{y}\t{'+-'[k & 1]}\t{'+-'[k >> 1]}\n"
              for i, (a, x, b, y, k) in enumerate(zip(c1.tolist(), p1.tolist(), c2.tolist(), p2.tolist(), s.tolist()))]
    return "".join(lines).encode()


def cases(seed=0):
    """name -> BGZF bytes of every kind of member the decoder must match zlib on"""
    rng = np.random.default_rng(seed)
    text = pairs_text(6000, seed)
    rand = rng.integers(0, 256, 3 * BLOCK, dtype=np.uint8).tobytes()
    far = rand[:32768] + rand[:BLOCK - 32768]                          # matches at distance 32 768
    out = {f"level{lv}": bgzf(text, level=lv) for lv in (0, 1, 6, 9)}
    for name, st in (("fixed", zlib.Z_FIXED), ("huffman_only", zlib.Z_HUFFMAN_ONLY), ("rle", zlib.Z_RLE), ("filtered", zlib.Z_FILTERED)):
        out[name] = bgzf(text, strategy=st)
    out["sync_flush"] = bgzf(text, flush=zlib.Z_SYNC_FLUSH, flush_every=1000)
    out["full_flush"] = bgzf(text, flush=zlib.Z_FULL_FLUSH, flush_every=777, level=9)
    out["random"] = bgzf(rand) + bgzf(rand[:5000], level=0)
    out["one_byte"] = bgzf(b"A" * (2 * BLOCK)) + bgzf(b"\n" * 300, strategy=zlib.Z_RLE)
    out["distance_32768"] = bgzf(far, level=9) + bgzf(far, level=1)
    out["sizes"] = b"".join(member(text[:k], level=lv) for k in (0, 1, 17, 4095, BLOCK) for lv in (0, 6)) + EOF
    out["foreign_subfield"] = b"".join(member(text[p:p + 3000], foreign=b"XY\x03\0abc") for p in range(0, 30000, 3000)) + EOF
    out["eof_only"] = EOF
    return out
