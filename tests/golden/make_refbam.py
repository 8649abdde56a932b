"""Writes tests/golden/refbam/ from the reference's own test BAMs (src/tests/data of the reference tree, located like
oracle/pyref/harness.py does): BAM files and CSI indices written by htslib, which tests/test_bamio.py reads back.

hg002.bam and hg002.bam.csi are copied unchanged.  hg008.bam (1.7 MB) is cut to its header and the records listed in KEEP: each
run of kept records fills whole BGZF blocks of the original, and those blocks are copied byte for byte, so every DEFLATE stream
in the cut is the one htslib wrote.  Its hg008.bam.csi is htslib's index with every virtual offset moved to where the kept
bytes now lie and the chunks of the dropped records removed.  Run where the reference tree exists:

    python tests/golden/make_refbam.py
"""
import os
import shutil
import struct
import sys
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle", "pyref")]
from sniffles_b200 import bamio  # noqa: E402
import harness  # noqa: E402

OUT = os.path.join(HERE, "refbam")
# hg008.bam: record 3 (chr1, spans two blocks) and records 12-13 (chrX, both in one block: the second starts mid-block)
KEEP = [3, 12, 13]


def _records(f):
    """(ref_id, first virtual offset, end virtual offset) of every record in file order"""
    out, v = [], f.first_record
    while True:
        d, v2 = f.bgzf.read_from(v, 4)
        if len(d) < 4:
            return out
        b, v3 = f.bgzf.read_from(v2, struct.unpack("<i", d)[0])
        out.append((struct.unpack("<i", b[:4])[0], v, v3))
        v = v3


def _read_csi(path):
    z = open(path, "rb").read()
    d, o = b"", 0
    while o < len(z):
        dec = zlib.decompressobj(31)
        d += dec.decompress(z[o:])
        o = len(z) - len(dec.unused_data)
    min_shift, depth, l_aux = struct.unpack("<iii", d[4:16])
    p = 16 + l_aux
    head = d[:p]
    n_ref = struct.unpack("<i", d[p:p + 4])[0]
    p += 4
    refs = []
    for _ in range(n_ref):
        n_bin = struct.unpack("<i", d[p:p + 4])[0]
        p += 4
        bins = []
        for _ in range(n_bin):
            b, lo, n_chunk = struct.unpack("<IQi", d[p:p + 16])
            p += 16
            bins.append((b, lo, [struct.unpack("<QQ", d[p + 16 * k:p + 16 * k + 16]) for k in range(n_chunk)]))
            p += 16 * n_chunk
        refs.append(bins)
    return head, refs, d[p:]


def cut_hg008(src, dst):
    f = bamio.BamFile(src)
    recs = _records(f)
    f.close()
    z = open(src, "rb").read()
    # runs of consecutive kept records, each [first block, end block) of the original file
    runs = []
    for i in KEEP:
        rid, v0, v1 = recs[i]
        assert v0 & 0xffff == 0 or (runs and runs[-1][1] == i), f"record {i} starts inside a block that also holds a dropped record"
        if runs and runs[-1][1] == i:
            runs[-1][1] = i + 1
        else:
            runs.append([i, i + 1])
    pieces = [(0, recs[0][1] >> 16)]                     # the header blocks
    for a, b in runs:
        end = recs[b - 1][2]
        assert end & 0xffff == 0, f"record {b - 1} ends inside a block that also holds a dropped record"
        pieces.append((recs[a][1] >> 16, end >> 16))
    eof = len(z) - len(bamio._BGZF_EOF)
    assert z[eof:] == bamio._BGZF_EOF
    pieces.append((eof, len(z)))
    new_start, o = [], 0
    for a, b in pieces:
        new_start.append(o)
        o += b - a

    def move(v):
        c, u = v >> 16, v & 0xffff
        for (a, b), s in zip(pieces, new_start):
            if a <= c <= b:
                return ((s + c - a) << 16) | u
        raise ValueError(f"virtual offset {c}:{u} lies in dropped bytes")
    with open(dst, "wb") as out:
        for a, b in pieces:
            out.write(z[a:b])

    kept = [(recs[i][0], recs[i][1], recs[i][2]) for i in KEEP]
    head, refs, tail = _read_csi(src + ".csi")
    body = bytearray(head + struct.pack("<i", len(refs)))
    for rid, bins in enumerate(refs):
        mine = [(v0, v1) for r, v0, v1 in kept if r == rid]
        entries = []
        for b, lo, chunks in bins:
            if b == 37450:                               # pseudo-bin: (first, end) offsets of the contig's records, (mapped, unmapped)
                if mine:
                    entries.append((b, lo, [(move(mine[0][0]), move(mine[-1][1])), (len(mine), 0)]))
                continue
            new = []
            for c0, c1 in chunks:
                for v0, v1 in mine:
                    if c0 <= v0 and v1 <= c1:
                        if new and new[-1][1] == move(v0):
                            new[-1] = (new[-1][0], move(v1))
                        else:
                            new.append((move(v0), move(v1)))
            if new:
                entries.append((b, min(move(v0) for v0, _ in mine if v0 >= lo), new))
        body += struct.pack("<i", len(entries))
        for b, lo, chunks in entries:
            body += struct.pack("<IQi", b, lo, len(chunks)) + b"".join(struct.pack("<QQ", *c) for c in chunks)
    body += tail
    with open(dst + ".csi", "wb") as out:
        for k in range(0, len(body), 0xff00):
            out.write(bamio._bgzf_block(bytes(body[k:k + 0xff00])))
        out.write(bamio._BGZF_EOF)


def main():
    data = os.path.join(harness.REFERENCE_SRC, "tests", "data")
    os.makedirs(OUT, exist_ok=True)
    for name in ("hg002.bam", "hg002.bam.csi"):
        shutil.copyfile(os.path.join(data, name), os.path.join(OUT, name))
    cut_hg008(os.path.join(data, "hg008.bam"), os.path.join(OUT, "hg008.bam"))


if __name__ == "__main__":
    main()
