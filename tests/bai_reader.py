"""A .bai reader and the standard region query, written from SAMv1 §5 for the tests of `sam2bam` (samtools is not in this image):
parse(bai) -> index; query_chunks(index, tid, beg, end) -> the chunks a reader visits for [beg, end); and a BAM walker that maps
virtual offsets to the records of the decompressed stream."""
import struct
import zlib

PSEUDO_BIN = 37450


def parse(bai):
    assert bai[:4] == b"BAI\1"
    n_ref, = struct.unpack_from("<i", bai, 4)
    p, refs = 8, []
    for _ in range(n_ref):
        n_bin, = struct.unpack_from("<i", bai, p); p += 4
        bins, pseudo = {}, None
        for _ in range(n_bin):
            b, n_chunk = struct.unpack_from("<Ii", bai, p); p += 8
            chunks = [struct.unpack_from("<QQ", bai, p + 16 * k) for k in range(n_chunk)]; p += 16 * n_chunk
            assert b not in bins and not (b == PSEUDO_BIN and pseudo), "a bin listed twice"
            if b == PSEUDO_BIN:
                assert n_chunk == 2
                pseudo = {"beg": chunks[0][0], "end": chunks[0][1], "n_mapped": chunks[1][0], "n_unmapped": chunks[1][1]}
            else:
                bins[b] = chunks
        n_intv, = struct.unpack_from("<i", bai, p); p += 4
        linear = list(struct.unpack_from(f"<{n_intv}Q", bai, p)); p += 8 * n_intv
        refs.append({"bins": bins, "pseudo": pseudo, "linear": linear})
    n_no_coor, = struct.unpack_from("<Q", bai, p); p += 8
    assert p == len(bai), "bytes after n_no_coor"
    return {"refs": refs, "n_no_coor": n_no_coor}


def bin_order(bai):
    """the bin numbers of every reference in file order (to check that they ascend)"""
    n_ref, = struct.unpack_from("<i", bai, 4)
    p, out = 8, []
    for _ in range(n_ref):
        n_bin, = struct.unpack_from("<i", bai, p); p += 4
        order = []
        for _ in range(n_bin):
            b, n_chunk = struct.unpack_from("<Ii", bai, p); p += 8 + 16 * n_chunk
            order.append(b)
        n_intv, = struct.unpack_from("<i", bai, p); p += 4 + 8 * n_intv
        out.append(order)
    return out


def reg2bins(beg, end):
    """every bin that may hold a record overlapping [beg, end) (SAMv1 §5.3)"""
    end -= 1
    out = [0]
    for shift, base in ((26, 1), (23, 9), (20, 73), (17, 585), (14, 4681)):
        out += range(base + (beg >> shift), base + (end >> shift) + 1)
    return out


def query_chunks(index, tid, beg, end):
    """the chunks of the bins of [beg, end), less those that end before the linear index's offset for beg"""
    r = index["refs"][tid]
    lin = r["linear"]
    min_off = lin[min(beg >> 14, len(lin) - 1)] if lin and (beg >> 14) < len(lin) else (lin[-1] if lin else 0)
    out = []
    for b in reg2bins(beg, end):
        for c in r["bins"].get(b, []):
            if c[1] > min_off:
                out.append(c)
    return sorted(out)


class BamFile:
    """the decompressed stream of a BAM file, with the file offset of every member, so that a virtual offset can be resolved"""

    def __init__(self, data):
        self.coff, self.uoff, parts, p, u = [], [], [], 0, 0
        while p < len(data):
            bsize, = struct.unpack_from("<H", data, p + 16)
            isize, = struct.unpack_from("<I", data, p + bsize + 1 - 4)
            self.coff.append(p); self.uoff.append(u)
            parts.append(zlib.decompress(data[p + 18:p + bsize + 1 - 8], -15))
            assert len(parts[-1]) == isize
            p += bsize + 1; u += isize
        self.coff.append(p); self.uoff.append(u)
        self.isizes = [len(x) for x in parts]
        self.raw = b"".join(parts)
        l_text, = struct.unpack_from("<i", self.raw, 4)
        q = 8 + l_text
        n_ref, = struct.unpack_from("<i", self.raw, q); q += 4
        self.refs = []
        for _ in range(n_ref):
            ln, = struct.unpack_from("<i", self.raw, q)
            self.refs.append((self.raw[q + 4:q + 4 + ln - 1].decode(), struct.unpack_from("<i", self.raw, q + 4 + ln)[0]))
            q += 8 + ln
        self.text = self.raw[8:8 + l_text].decode()
        self.rec_start = q
        self.records = []                                   # (uncompressed offset, bytes)
        while q < len(self.raw):
            n, = struct.unpack_from("<I", self.raw, q)
            self.records.append((q, self.raw[q:q + 4 + n])); q += 4 + n
        self.by_off = {o: k for k, (o, _) in enumerate(self.records)}
        self.coff_index = {c: k for k, c in enumerate(self.coff)}

    def resolve(self, voff):
        """virtual offset -> uncompressed offset"""
        k = self.coff_index[voff >> 16]
        assert (voff & 0xffff) <= (self.isizes[k] if k < len(self.isizes) else 0)
        return self.uoff[k] + (voff & 0xffff)

    def records_in(self, chunk):
        """the records a reader reads from a chunk"""
        a, b = self.resolve(chunk[0]), self.resolve(chunk[1])
        k = self.by_off[a]
        out = []
        while k < len(self.records) and self.records[k][0] < b:
            out.append(k); k += 1
        return out


def rec_fields(rec):
    tid, pos = struct.unpack_from("<ii", rec, 4)
    bin_, = struct.unpack_from("<H", rec, 14)
    l_name, n_cig, flag = rec[12], struct.unpack_from("<H", rec, 16)[0], struct.unpack_from("<H", rec, 18)[0]
    ln = 0
    for k in range(n_cig):
        v, = struct.unpack_from("<I", rec, 36 + l_name + 4 * k)
        if v & 15 in (0, 2, 3, 7, 8):
            ln += v >> 4
    end = pos + (1 if flag & 4 or ln == 0 else ln)
    return tid, pos, end, bin_, flag
