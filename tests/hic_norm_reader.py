"""Independent reader of the normalised section of a `.hic` version 8 file, written from the published format description:
header -> master index position -> footer (nBytesV5 skips the master index and the raw expected values) -> normalised
expected values -> normalisation vector index -> the vectors at their file positions.  Test infrastructure for the vectors
csrc/hic_writer.hpp stores (`pairs2bins -n`); shares no code with the writer or with tests/hic_reader.py."""
import struct


def _cstr(data, p):
    e = data.index(b"\0", p)
    return data[p:e].decode(), e + 1


def read_norm(path):
    """-> dict(chroms [(name, len)], resolutions, master_pos, n_bytes_v5, section_start,
    expected {(type, bin_size): (values, {chr: scale})}, vectors {(type, chr, bin_size): [values]},
    index [(type, chr, bin_size, position, n_bytes)] in file order)"""
    data = open(path, "rb").read()
    assert data[:4] == b"HIC\0" and struct.unpack_from("<i", data, 4)[0] == 8
    master_pos = struct.unpack_from("<q", data, 8)[0]
    p = 16
    _, p = _cstr(data, p)                                            # genome id
    (n_attr,) = struct.unpack_from("<i", data, p); p += 4
    for _ in range(2 * n_attr):
        _, p = _cstr(data, p)
    (n_chr,) = struct.unpack_from("<i", data, p); p += 4
    chroms = []
    for _ in range(n_chr):
        name, p = _cstr(data, p)
        (ln,) = struct.unpack_from("<i", data, p); p += 4
        chroms.append((name, ln))
    (n_res,) = struct.unpack_from("<i", data, p); p += 4
    resolutions = list(struct.unpack_from("<%di" % n_res, data, p))

    (n_bytes_v5,) = struct.unpack_from("<i", data, master_pos)
    p = master_pos + 4 + n_bytes_v5
    out = {"chroms": chroms, "resolutions": resolutions, "master_pos": master_pos, "n_bytes_v5": n_bytes_v5, "section_start": p,
           "expected": {}, "vectors": {}, "index": []}
    (n_exp,) = struct.unpack_from("<i", data, p); p += 4
    for _ in range(n_exp):
        typ, p = _cstr(data, p)
        unit, p = _cstr(data, p)
        assert unit == "BP"
        bs, nv = struct.unpack_from("<ii", data, p); p += 8
        vals = list(struct.unpack_from("<%dd" % nv, data, p)); p += 8 * nv
        (ns,) = struct.unpack_from("<i", data, p); p += 4
        scale = {}
        for _ in range(ns):
            ci, sc = struct.unpack_from("<id", data, p); p += 12
            scale[ci] = sc
        assert (typ, bs) not in out["expected"]
        out["expected"][(typ, bs)] = (vals, scale)
    (n_vec,) = struct.unpack_from("<i", data, p); p += 4
    for _ in range(n_vec):
        typ, p = _cstr(data, p)
        (ci,) = struct.unpack_from("<i", data, p); p += 4
        unit, p = _cstr(data, p)
        assert unit == "BP"
        bs, pos, nb = struct.unpack_from("<iqi", data, p); p += 16
        out["index"].append((typ, ci, bs, pos, nb))
    end = p
    for typ, ci, bs, pos, nb in out["index"]:
        (nv,) = struct.unpack_from("<i", data, pos)
        assert nb == 4 + 8 * nv, "nBytes = 4 + 8 nValues"
        assert (typ, ci, bs) not in out["vectors"]
        out["vectors"][(typ, ci, bs)] = list(struct.unpack_from("<%dd" % nv, data, pos + 4))
        end = max(end, pos + nb)
    # the vectors lie back to back right behind the index, and the file ends after the last one
    pos = p
    for _, _, _, vp, nb in sorted(out["index"], key=lambda e: e[3]):
        assert vp == pos, "vectors back to back after the index"
        pos += nb
    assert end == len(data) and pos == len(data)
    return out
