"""BGZF / BAM / BAI stand-in for htslib (SURVEY 8a row A0): a block written as BAM + BAI and fetched back by region equals the block."""
import os

import numpy as np
import pytest

from sniffles_b200 import abi, bamio, synth


@pytest.fixture(scope="module")
def bam(tmp_path_factory):
    blk = synth.generate(31, [300_000, 180_000], 12.0, len_mean=9000.0, len_sd=2500.0, sv_spacing=5000.0, phased_frac=0.5)
    path = str(tmp_path_factory.mktemp("bam") / "t.bam")
    bamio.write_bam(path, blk)
    return blk, path


def _key(r):
    return (r["pos"], r["flag"], r["mapq"], r["l_seq"], bytes(r["qname"]), r["cigar"].tobytes(), r["seq"].tobytes(), r["aux"].get("NM"), r["aux"].get("SA"), r["aux"].get("HP"), r["aux"].get("PS"))


def _block_records(blk, t):
    out = []
    for r in blk.rec[blk.rec["task"] == t]:
        co, n = int(r["cigar_off"]), int(r["n_cigar"])
        vo, lq, sl = int(r["var_off"]), int(r["l_qname"]), int(r["sa_len"])
        so, ls = int(r["seq_off"]), int(r["l_seq"])
        af = int(r["aux_flags"])
        out.append((int(r["pos"]), int(r["flag"]), int(r["mapq"]), ls, bytes(blk.var[vo:vo + lq]), blk.cigar[co:co + n].tobytes(), blk.seq[so:so + (ls + 1) // 2].tobytes(),
                    int(r["nm"]) if af & abi.AUX_NM else None, bytes(blk.var[vo + lq:vo + lq + sl]) if af & abi.AUX_SA else None,
                    int(r["hp"]) if af & abi.AUX_HP else None, int(r["ps"]) if af & abi.AUX_PS else None))
    return out


def test_whole_contig_fetch_round_trips(bam):
    blk, path = bam
    f = bamio.BamFile(path)
    assert [n for n, _ in f.contigs] == blk.contig_names
    for t, name in enumerate(blk.contig_names):
        got = [_key(r) for r in f.fetch(name, 0, f.get_reference_length(name))]
        assert got == _block_records(blk, t)
        assert f.count_mapped(name) == len(got)
    f.close()


def test_region_fetch_equals_overlap_filter(bam):
    blk, path = bam
    f = bamio.BamFile(path)
    rnd = np.random.default_rng(3)
    for _ in range(20):
        t = int(rnd.integers(0, 2))
        L = f.get_reference_length(blk.contig_names[t])
        a = int(rnd.integers(0, L - 1000)); b = a + int(rnd.integers(1, 60000))
        got = [_key(r) for r in f.fetch(blk.contig_names[t], a, b)]
        want = []
        for r, k in zip(blk.rec[blk.rec["task"] == t], _block_records(blk, t)):
            span = bamio.ref_span(blk.cigar[int(r["cigar_off"]):int(r["cigar_off"]) + int(r["n_cigar"])])
            if k[0] < b and k[0] + max(span, 1) > a:
                want.append(k)
        assert got == want, (t, a, b)
    f.close()


def test_long_cigar_escape(tmp_path):
    """more than 65535 CIGAR ops: the CG:B,I tag carries the real CIGAR behind an <l_seq>S<reflen>N placeholder"""
    n = 70000
    cig = np.empty(n, "<u4"); cig[0::2] = (3 << 4) | 0; cig[1::2] = (1 << 4) | 2          # 3M 1D ...
    l_seq = 3 * (n // 2)
    rec = np.zeros(1, abi.REC_DTYPE)
    rec[0] = (0, 100, 0, 60, abi.AUX_NM, 0, 2, 0, 5, 0, n, l_seq, 0, 0, 0, 0, 0)
    contig = np.zeros(1, abi.CONTIG_DTYPE); contig[0] = (abi.fnv1a64(b"c"), 1_000_000, 0)
    task = np.zeros(1, abi.TASK_DTYPE); task[0] = (0, 0, 999_999, 1_000_000, 0, 0, 0, 0)
    blk = synth.RecordBlock(rec=rec, cigar=cig, var=np.frombuffer(b"rd", "u1"), seq=np.full((l_seq + 1) // 2, 0x12, "u1"), task=task, contig=contig, tr=np.zeros(0, "<i4"), contig_names=["c"])
    path = str(tmp_path / "long.bam")
    bamio.write_bam(path, blk)
    f = bamio.BamFile(path)
    rs = list(f.fetch("c", 0, 1_000_000))
    assert len(rs) == 1 and len(rs[0]["cigar"]) == n and (rs[0]["cigar"] == cig).all()
    f.close()


def test_csi_index_equals_bai(bam, tmp_path):
    """the same records through a CSI index (BGZF-compressed, per-bin loffsets instead of the linear index) — the reference's own test
    BAMs carry .csi indices"""
    blk, path = bam
    p2 = str(tmp_path / "c.bam")
    bamio.write_bam(p2, blk, index="csi")
    fa, fb = bamio.BamFile(path), bamio.BamFile(p2)
    assert fb.index[0][1] is None and fb.index[0][2] and fa.index[0][1] is not None
    rnd = np.random.default_rng(2)
    for _ in range(40):
        t = int(rnd.integers(0, 2))
        L = fa.get_reference_length(blk.contig_names[t])
        a = int(rnd.integers(0, L - 10)); b = a + int(rnd.integers(1, 80000))
        assert [_key(r) for r in fa.fetch(blk.contig_names[t], a, b)] == [_key(r) for r in fb.fetch(blk.contig_names[t], a, b)]
        assert fa.merged_chunks(blk.contig_names[t], a, b) and fb.merged_chunks(blk.contig_names[t], a, b)
    for n in blk.contig_names:
        assert fa.count_mapped(n) == fb.count_mapped(n)
    fa.close(); fb.close()


REF_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "refbam")


@pytest.mark.parametrize("name", ["hg008.bam", "hg002.bam"])
def test_reference_bams_through_csi_and_device_spans(name):
    """htslib-written files (the reference's test BAMs; hg008.bam cut to three of its records by tests/golden/make_refbam.py, its
    blocks unchanged): region fetch through their .csi equals a linear scan, the one-lane host build of the device DEFLATE decoder
    inflates every block like zlib, and the spans of device_input cover exactly the records of every contig"""
    import struct
    import zlib
    import ingest_emul
    f = bamio.BamFile(os.path.join(REF_DATA, name))
    v, allr = f.first_record, []
    while True:
        d, v2 = f.bgzf.read_from(v, 4)
        if len(d) < 4:
            break
        b, v = f.bgzf.read_from(v2, struct.unpack("<i", d)[0])
        r = bamio.decode_record(b)
        if r["ref_id"] >= 0:
            allr.append(r)
    assert allr
    z = open(os.path.join(REF_DATA, name), "rb").read()
    for k, (_, po, pl, isz) in enumerate(ingest_emul.walk_bgzf(z)):
        rc, got = ingest_emul.inflate(z[po:po + pl], isz, lead=k % 4)
        assert rc == 0 and got == zlib.decompress(z[po:po + pl], -15)
    key = lambda r: (r["pos"], bytes(r["qname"]), r["flag"])
    rnd = np.random.default_rng(1)
    for rid in sorted({r["ref_id"] for r in allr}):
        rs = [r for r in allr if r["ref_id"] == rid]
        cname, L = f.contigs[rid]
        lo, hi = min(r["pos"] for r in rs), max(r["pos"] + max(bamio.ref_span(r["cigar"]), 1) for r in rs)
        for _ in range(20):
            a = int(rnd.integers(max(lo - 50000, 0), hi)); b = a + int(rnd.integers(1, 200000))
            assert [key(r) for r in f.fetch(cname, a, b)] == [key(r) for r in rs if r["pos"] < b and r["pos"] + max(bamio.ref_span(r["cigar"]), 1) > a]
        task = np.zeros(1, abi.TASK_DTYPE); task[0] = (rid, 0, L, L, 0, 0, 0, 0)
        bg, sp = f.device_input([(cname, 0, L)])
        assert [(d["pos"], d["qname"], d["flag"]) for d in ingest_emul.load_bam(bg, sp, task)] == [key(r) for r in rs]
    f.close()
