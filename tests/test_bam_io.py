"""host/bam.cpp (the SAM / BAM reader and BGZF writer behind rsem-run-em -b) on CPU, through bin/rsem-b200-host-selftest:
SAM -> BAM conversion against an independent decode of the SAM text, BAM -> BAM copy, MAPQ / ZW:f as the reference sets
them (BamWriter.h:39-48, sam_utils.h:72-76), for several compression thread counts."""
import math
import os
import subprocess

import numpy as np
import pytest

import ref_golden
import rsem_files as rf
from bam_reader import read_bam

EXE = os.path.join(rf.ROOT, "bin", "rsem-b200-host-selftest")


def _sam_records(path):
    hdr, recs = [], []
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            if line.startswith("@"):
                hdr.append(line)
                continue
            t = line.split("\t")
            recs.append(dict(qname=t[0], flag=int(t[1]), rname=t[2], pos=int(t[3]) - 1, mapq=int(t[4]), cigar=t[5], rnext=t[6],
                             mpos=int(t[7]) - 1, tlen=int(t[8]), seq=t[9], qual=t[10], extra=t[11:]))
    return hdr, recs


def _mapq(p):
    err = 1.0 - p
    return 100 if err <= 1e-10 else int(-10 * math.log10(err) + .5)


@pytest.mark.parametrize("read_type,threads", [(1, 1), (3, 4), (0, 2)])
def test_sam_to_bam_and_weights(tmp_path, built, read_type, threads):
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=read_type, M=40, N1=700, N0=60, read_len=45, sam=1, seed=read_type + 1)
    # a few optional fields of every type on the first alignment lines (the converter must encode them like htslib)
    lines = open(f"{d}/aln.sam").read().split("\n")
    k = next(i for i, l in enumerate(lines) if l and not l.startswith("@"))
    lines[k] += "\tNM:i:3\tXA:A:Q\tXS:i:-70000\tXF:f:2.5\tXZ:Z:hello world\tXB:B:s,-3,4,500\tZW:f:0.25\tXU:i:70000\tXH:H:1AE3"
    open(f"{d}/aln2.sam", "w").write("\n".join(lines))
    step = 0.0137
    out = subprocess.check_output([EXE, "--bam-copy", f"{d}/aln2.sam", f"{d}/out.bam", str(threads), str(step)], text=True)
    hdr, sam = _sam_records(f"{d}/aln2.sam")
    text, refs, bam = read_bam(f"{d}/out.bam")
    assert f"records {len(sam)} " in out and len(bam) == len(sam)
    assert text == "\n".join(hdr) + "\n@PG\tID:RSEM\n"   # SamHeader regroups HD, SQ, RG, PG (+ RSEM), CO
    names = [n for n, _ in refs]
    assert names == [h.split("\t")[1][3:] for h in hdr if h.startswith("@SQ")]
    mapped = 0
    for s, b in zip(sam, bam):
        assert (b["qname"], b["flag"], b["pos"], b["cigar"], b["mpos"], b["tlen"], b["seq"]) == \
               (s["qname"], s["flag"], s["pos"], s["cigar"], s["mpos"], s["tlen"], s["seq"])
        assert b["qual"] == s["qual"]
        assert b["tid"] == (-1 if s["rname"] == "*" else names.index(s["rname"]))
        if s["flag"] & 4:
            assert b["mapq"] == s["mapq"] and "ZW" not in b["tags"]
        else:
            mapped += 1
            p = (mapped * step) % 1.0
            assert b["mapq"] == _mapq(p)
            assert b["tags"]["ZW"][0] == "f" and abs(b["tags"]["ZW"][1] - p) <= 1e-7
    t = bam[0]["tags"]
    assert t["NM"] == ("i", 3) and t["XA"] == ("A", "Q") and t["XS"] == ("i", -70000) and t["XU"] == ("i", 70000)
    assert t["XF"] == ("f", 2.5) and t["XZ"] == ("Z", "hello world") and t["XB"] == ("B", ("s", [-3, 4, 500])) and t["XH"] == ("H", "1AE3")
    # BAM in -> BAM out, no weights: records unchanged
    subprocess.check_call([EXE, "--bam-copy", f"{d}/out.bam", f"{d}/copy.bam", "3"], stdout=subprocess.DEVNULL)
    text2, refs2, bam2 = read_bam(f"{d}/copy.bam")
    assert refs2 == refs and bam2 == bam and text2 == text   # RSEM's @PG is not added twice
    # the BGZF stream ends with the EOF marker block
    assert open(f"{d}/copy.bam", "rb").read()[-28:] == bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 66, 67, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0])


def test_conversion_matches_htslib(tmp_path, built):
    """our SAM -> BAM encoding against htslib's (through the reference's own rsem-run-em -b): identical records apart from the
    posterior fields (MAPQ, ZW).  The reference's records are pinned by a digest in tests/golden/ref_outputs.json.gz
    (tools/make_golden_ref.py)."""
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=3, M=30, N1=300, N0=20, read_len=40, sam=1, seed=9)
    subprocess.check_call([EXE, "--bam-copy", f"{d}/aln.sam", f"{d}/ours.bam", "2"], stdout=subprocess.DEVNULL)
    ours = ref_golden.bam_outputs(f"{d}/ours.bam")
    assert np.isnan(ours["zw"]).all()
    assert ref_golden.Run("bam_io/htslib").same(ours, "records")
