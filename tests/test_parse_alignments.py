"""bin/rsem-parse-alignments (rsem_b200/host/main_parse.cpp) and the binary side-car it hands to rsem-run-em - CPU only.

Reference behaviour: the reference's parseIt.cpp:64-229, SamParser.h:97-265, Transcripts.h:105-143.
  * every output file (.dat, the read files per category, .cnt, .omit) is BYTE-IDENTICAL to what the reference's
    rsem-parse-alignments (oracle/_ref, built from the reference sources with its vendored htslib) writes, for all four
    read types, SAM and BAM input, and with the aligner's "too many alignments" tag (-tag, the N2 category): the
    reference's files are pinned by their SHA-256 in tests/golden/ref_outputs.json.gz (tools/make_golden_ref.py);
  * imd.b200 holds the same hits and reads as the text files: compared array by array with what the text parsers of
    rsem-run-em produce from the files next to it (rsem-b200-host-selftest dumps both), including the low-quality flags
    and the names of the reads shorter than the seed length; a stale side-car (text file replaced) is refused.
"""
import filecmp
import os
import subprocess

import numpy as np
import pytest

import ref_golden
import rsem_files as rf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OURS = os.path.join(ROOT, "bin", "rsem-parse-alignments")
SELFTEST = os.path.join(ROOT, "bin", "rsem-b200-host-selftest")


def _parse(exe, d, aln, read_type, out, extra=()):
    os.makedirs(f"{out}/t", exist_ok=True)
    os.makedirs(f"{out}/s", exist_ok=True)
    p = subprocess.run([exe, f"{d}/ref/r", f"{out}/t/s", f"{out}/s/s", aln, str(read_type), "-q", *extra],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    return p


def _files(out):
    return sorted(os.path.join(dp, f)[len(out) + 1:] for dp, _, fs in os.walk(out) for f in fs if not f.endswith(".b200"))


def _assert_same_tree(a, b):
    fa, fb = _files(a), _files(b)
    assert fa == fb, (fa, fb)
    for f in fa:
        assert filecmp.cmp(os.path.join(a, f), os.path.join(b, f), shallow=False), f"{f} differs"


def _assert_same_as_reference(key, out):
    """the files in out are those the reference wrote in the stored run `key`, byte for byte"""
    g = ref_golden.Run(key)
    files = _files(out)
    assert "\n".join(files) == g["files"], (files, g["files"])
    for f in files:
        assert ref_golden.file_digest(os.path.join(out, f)) == g["file:" + f], f"{f} differs"


@pytest.mark.parametrize("read_type", [0, 1, 2, 3])
def test_outputs_byte_identical_to_the_reference(built, tmp_path, read_type):
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=read_type, M=150, N1=3000, N0=200, read_len=50, var_len=30, seed=5 + read_type,
                       sam=1, spurious=0.05, omit=7)
    sam = f"{d}/aln.sam"
    o = _parse(OURS, d, sam, read_type, str(tmp_path / "ours"))
    assert o.returncode == 0, o.stderr
    _assert_same_as_reference(f"parse/byte_identical/{read_type}/sam", str(tmp_path / "ours"))
    assert os.path.getsize(tmp_path / "ours" / "t" / "s.dat") > 1000
    # the reference's .dat equals the generator's hand-written one up to the padded header line (SURVEY 8(c))
    # BAM input (converted by this repository's own BGZF writer): same files again, from both programs
    bam = str(tmp_path / "aln.bam")
    subprocess.check_call([SELFTEST, "--bam-copy", sam, bam, "2"], stdout=subprocess.DEVNULL)
    ob = _parse(OURS, d, bam, read_type, str(tmp_path / "ours_bam"))
    assert ob.returncode == 0, ob.stderr
    _assert_same_as_reference(f"parse/byte_identical/{read_type}/bam", str(tmp_path / "ours_bam"))
    for f in _files(str(tmp_path / "ours")):
        if f.endswith(".dat") or f.endswith(".cnt") or ".f" in f:   # .omit differs only if the header differs: it does not
            assert filecmp.cmp(tmp_path / "ours" / f, tmp_path / "ours_bam" / f, shallow=False), f


def _tag_some_unaligned(sam_in, sam_out, paired):
    """gives every third unaligned read (pair) the bowtie tag XM:i:2 -> category N2 ("max") with -tag XM; one gets XM:i:0"""
    k = 0
    with open(sam_in) as fi, open(sam_out, "w") as fo:
        lines = fi.readlines()
        i = 0
        while i < len(lines):
            ln = lines[i]
            if ln.startswith("@"):
                fo.write(ln); i += 1
                continue
            n = 2 if paired else 1
            grp = lines[i:i + n]
            if int(grp[0].split("\t")[1]) & 4:
                k += 1
                if k % 3 == 0:
                    val = 0 if k % 9 == 0 else 2
                    grp = [g.rstrip("\n") + f"\tXM:i:{val}\n" for g in (grp if k % 2 else grp[-1:])] if not paired or k % 2 else \
                          [grp[0], grp[1].rstrip("\n") + f"\tXM:i:{val}\n"]
            fo.writelines(grp)
            i += n
    return sam_out


@pytest.mark.parametrize("read_type", [1, 2])
def test_too_many_alignments_tag(built, tmp_path, read_type):
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=read_type, M=80, N1=1500, N0=400, read_len=40, seed=3, sam=1)
    sam = _tag_some_unaligned(f"{d}/aln.sam", str(tmp_path / "tagged.sam"), read_type >= 2)
    o = _parse(OURS, d, sam, read_type, str(tmp_path / "ours"), ("-tag", "XM"))
    assert o.returncode == 0, o.stderr
    _assert_same_as_reference(f"parse/tag/{read_type}", str(tmp_path / "ours"))
    n0, n1, n2, tot = (int(x) for x in open(tmp_path / "ours" / "s" / "s.cnt").readline().split())
    assert n2 > 50 and n0 > 50 and n0 + n1 + n2 == tot
    assert any(f.startswith("t/s_max") for f in _files(str(tmp_path / "ours")))


def test_errors_follow_the_reference_convention(built, tmp_path):
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=0, M=30, N1=200, N0=20, read_len=40, seed=1, sam=1)
    p = subprocess.run([OURS], stdout=subprocess.PIPE, text=True)
    assert p.returncode == 255 and p.stdout.startswith("Usage : rsem-parse-alignments refName imdName statName alignF read_type")
    # a paired-end flag in single-end mode: message on stderr, exit(-1) (SamParser.h:110)
    bad = str(tmp_path / "bad.sam")
    lines = open(f"{d}/aln.sam").read().split("\n")
    k = next(i for i, l in enumerate(lines) if l and not l.startswith("@"))
    f = lines[k].split("\t")
    f[1] = str(int(f[1]) | 1)
    lines[k] = "\t".join(f)
    open(bad, "w").write("\n".join(lines))
    p = _parse(OURS, d, bad, 0, str(tmp_path / "o"))
    assert p.returncode == 255 and "Find a paired end read in the file!" in p.stderr
    p = _parse(OURS, d, str(tmp_path / "missing.sam"), 0, str(tmp_path / "o2"))
    assert p.returncode == 255 and "It may not exist" in p.stderr


@pytest.mark.parametrize("read_type", [1, 3])
def test_sidecar_equals_the_text_files(built, tmp_path, read_type):
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=read_type, M=120, N1=4000, N0=300, read_len=50, var_len=35, seed=11, sam=1,
                       polyA=20)
    out = str(tmp_path / "o")
    assert _parse(OURS, d, f"{d}/aln.sam", read_type, out).returncode == 0
    imd = f"{out}/t/s"
    assert os.path.exists(imd + ".b200")
    seed_len = 25
    txt, sc = str(tmp_path / "txt"), str(tmp_path / "sc")
    subprocess.check_call([SELFTEST, imd, str(read_type), "3", str(seed_len), txt], stdout=subprocess.DEVNULL)
    p = subprocess.run([SELFTEST, "--sidecar", imd, str(read_type), "3", str(seed_len), "0", sc], stdout=subprocess.PIPE, text=True)
    assert p.returncode == 0, p.stdout
    names = ["row_ptr.u64", "sid.i32", "pos.i32", "lowq.u8", "off0.u64", "base0.u8", "qual0.u8"]
    if read_type >= 2:
        names += ["insertL.i32", "off1.u64", "base1.u8", "qual1.u8"]
    for n in names:
        a, b = np.fromfile(f"{txt}.{n}", np.uint8), np.fromfile(f"{sc}.{n}", np.uint8)
        assert len(a) > 0 and np.array_equal(a, b), n
    lowq = np.fromfile(f"{sc}.lowq.u8", np.uint8)
    assert 0 < lowq.sum() < len(lowq)   # var_len 35: some reads are shorter than the seed length
    # the short-read names are the ones the text path reports (first 50, file order)
    short = [l.split()[2] for l in p.stdout.splitlines() if l.startswith("short 1 ")]
    ext = "fq"
    lines = open(f"{imd}_alignable{'_1' if read_type >= 2 else ''}.{ext}").read().split("\n")
    lines2 = open(f"{imd}_alignable_2.{ext}").read().split("\n") if read_type >= 2 else None
    want = []
    for r in range(len(lowq)):
        l1 = len(lines[4 * r + 1])
        l2 = len(lines2[4 * r + 1]) if lines2 else l1
        if min(l1, l2) < seed_len:
            want.append(lines[4 * r][1:])
    assert short == want[:50] and len(want) > 0
    # with a poly(A) reference the flags still agree with an independent evaluation (SingleReadQ.h:63-95)
    p = subprocess.run([SELFTEST, "--sidecar", imd, str(read_type), "2", str(seed_len), "1", sc + "A"], stdout=subprocess.PIPE, text=True)
    assert p.returncode == 0
    lowqA = np.fromfile(f"{sc}A.lowq.u8", np.uint8)
    ref_lq = []
    for r in range(len(lowq)):
        m1 = rf._single_lq(lines[4 * r + 1], True, seed_len)
        if lines2:
            s1, s2 = lines[4 * r + 1], lines2[4 * r + 1]
            lq = True if (len(s1) < seed_len or len(s2) < seed_len) else (m1 and rf._single_lq(s2, True, seed_len))
        else:
            lq = m1
        ref_lq.append(1 if lq else 0)
    assert np.array_equal(lowqA, np.array(ref_lq, np.uint8))
    # a side-car that no longer describes the text files is refused
    with open(imd + ".dat", "a") as f:
        f.write("\n")
    p = subprocess.run([SELFTEST, "--sidecar", imd, str(read_type), "1", str(seed_len), "0", sc + "X"], stdout=subprocess.PIPE, text=True)
    assert p.returncode == 3 and "no usable side-car" in p.stdout
    env = dict(os.environ, RSEM_B200_SIDECAR="0")
    out2 = str(tmp_path / "o2")
    os.makedirs(f"{out2}/t"); os.makedirs(f"{out2}/s")
    subprocess.check_call([OURS, f"{d}/ref/r", f"{out2}/t/s", f"{out2}/s/s", f"{d}/aln.sam", str(read_type), "-q"], env=env)
    assert not os.path.exists(f"{out2}/t/s.b200")


def test_sidecar_refused_when_dat_content_changes_at_equal_size(built, tmp_path):
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=0, M=60, N1=800, N0=50, read_len=40, seed=2, sam=1)
    out = str(tmp_path / "o")
    assert _parse(OURS, d, f"{d}/aln.sam", 0, out).returncode == 0
    imd = f"{out}/t/s"
    ok = subprocess.run([SELFTEST, "--sidecar", imd, "0", "1", "25", "0", str(tmp_path / "a")], stdout=subprocess.PIPE, text=True)
    assert ok.returncode == 0
    data = bytearray(open(imd + ".dat", "rb").read())
    k = data.rindex(b" ")          # change one digit of the last position: same size, other content
    data[k + 1] = ord("7") if data[k + 1] != ord("7") else ord("8")
    open(imd + ".dat", "wb").write(bytes(data))
    bad = subprocess.run([SELFTEST, "--sidecar", imd, "0", "1", "25", "0", str(tmp_path / "b")], stdout=subprocess.PIPE, text=True)
    assert bad.returncode == 3 and "no usable side-car" in bad.stdout


def test_reader_variants_give_the_same_files(built, tmp_path):
    """AlnReader (host/bam.cpp): plain SAM, gzip'ed SAM (one gzip member: zlib's gz layer), BAM = BGZF (blocks inflated on
    1 or 8 worker threads ahead of the parser) - the same output files every time; a truncated BAM is an error, not a
    short result."""
    import gzip
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=3, M=90, N1=6000, N0=300, read_len=45, seed=4, sam=1, spurious=0.02)
    sam = f"{d}/aln.sam"
    gz = str(tmp_path / "aln.sam.gz")
    with open(sam, "rb") as fi, gzip.open(gz, "wb", compresslevel=1) as fo:
        fo.write(fi.read())
    bam = str(tmp_path / "aln.bam")
    subprocess.check_call([SELFTEST, "--bam-copy", sam, bam, "3"], stdout=subprocess.DEVNULL)
    assert os.path.getsize(bam) > 10 * 65536 / 8   # several BGZF blocks
    outs = {}
    for tag, aln, env in (("sam", sam, {}), ("gz", gz, {}), ("bam1", bam, {"RSEM_B200_IO_THREADS": "1"}),
                          ("bam8", bam, {"RSEM_B200_IO_THREADS": "8"})):
        out = str(tmp_path / tag)
        os.makedirs(f"{out}/t"); os.makedirs(f"{out}/s")
        p = subprocess.run([OURS, f"{d}/ref/r", f"{out}/t/s", f"{out}/s/s", aln, "3", "-q"], env=dict(os.environ, **env),
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert p.returncode == 0, p.stderr
        outs[tag] = out
    for tag in ("gz", "bam1", "bam8"):
        _assert_same_tree(outs["sam"], outs[tag])
        assert open(outs[tag] + "/t/s.b200", "rb").read() == open(outs["sam"] + "/t/s.b200", "rb").read()
    # truncated in the middle of a block
    cut = str(tmp_path / "cut.bam")
    open(cut, "wb").write(open(bam, "rb").read()[: os.path.getsize(bam) // 2])
    out = str(tmp_path / "cut")
    os.makedirs(f"{out}/t"); os.makedirs(f"{out}/s")
    p = subprocess.run([OURS, f"{d}/ref/r", f"{out}/t/s", f"{out}/s/s", cut, "3", "-q"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert p.returncode == 255 and ("Truncated" in p.stderr or "Corrupt" in p.stderr or "corrupt" in p.stderr)


@pytest.mark.parametrize("name,read_type,extra", [("parse_pe_q", 3, ()), ("parse_se_noq_tag", 0, ("-tag", "XM"))])
def test_golden_outputs_of_the_reference(built, tmp_path, name, read_type, extra):
    """tests/golden/parse_*.tar.gz (tools/make_golden_parse.py): outputs of the reference's own rsem-parse-alignments; pins our
    program where oracle/_ref is not available.  SAM input and the BAM made from it."""
    import tarfile
    with tarfile.open(os.path.join(ROOT, "tests", "golden", name + ".tar.gz")) as tar:
        tar.extractall(tmp_path, filter="data")
    g = str(tmp_path / name)
    bam = str(tmp_path / "aln.bam")
    subprocess.check_call([SELFTEST, "--bam-copy", f"{g}/aln.sam", bam, "2"], stdout=subprocess.DEVNULL)
    for tag, aln in (("sam", f"{g}/aln.sam"), ("bam", bam)):
        out = str(tmp_path / tag)
        os.makedirs(f"{out}/t"); os.makedirs(f"{out}/s")
        p = subprocess.run([OURS, f"{g}/ref/r", f"{out}/t/s", f"{out}/s/s", aln, str(read_type), "-q", *extra],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert p.returncode == 0, p.stderr
        _assert_same_tree(f"{g}/out", out)


def test_damaged_sidecar_is_refused_not_trusted(built, tmp_path):
    d = rf.gen_dataset(str(tmp_path / "d"), read_type=1, M=60, N1=900, N0=60, read_len=40, seed=6, sam=1)
    out = str(tmp_path / "o")
    assert _parse(OURS, d, f"{d}/aln.sam", 1, out).returncode == 0
    imd = f"{out}/t/s"
    blob = bytearray(open(imd + ".b200", "rb").read())
    import struct
    for what, patch in (("huge H", lambda b: b.__setitem__(slice(40, 48), struct.pack("<Q", 1 << 60))),
                        ("truncated", lambda b: b.__delitem__(slice(len(b) // 2, len(b))))):
        bad = bytearray(blob)
        patch(bad)
        open(imd + ".b200", "wb").write(bytes(bad))
        p = subprocess.run([SELFTEST, "--sidecar", imd, "1", "1", "25", "0", str(tmp_path / "x")], stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True)
        assert p.returncode == 3 and "no usable side-car" in p.stdout, what
