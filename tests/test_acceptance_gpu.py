"""Drop-in acceptance test (SURVEY.md section 8(c)): the UNMODIFIED Perl driver rsem-calculate-expression runs the whole
pipeline - rsem-parse-alignments, rsem-build-read-index, rsem-run-em (with its default -b posterior BAM and --gibbs-out),
rsem-run-gibbs - once with the reference's binaries (oracle/_ref) and once with bin/rsem-run-em and bin/rsem-run-gibbs
(and bin/rsem-parse-alignments, whose binary side-car rsem-run-em then loads instead of parsing .dat and the read files)
swapped in beside the same driver.  Compared: *.isoforms.results, *.genes.results (EM and posterior-mean columns) and
every record of *.transcript.bam (MAPQ, ZW tag).  The driver, its module and the reference tools are installed into
oracle/_ref by oracle/Makefile; nothing is read from /root/reference at run time."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import rsem_files as rf
from bam_reader import read_bam

pytestmark = pytest.mark.gpu
DRIVER = os.path.join(rf.REF_DIR, "rsem-calculate-expression")


def _install(dst, which):
    """a bin directory as `make install` lays it out: the driver finds its tools beside itself (rsem-calculate-expression:12)"""
    os.makedirs(dst)
    for f in ("rsem-calculate-expression", "rsem_perl_utils.pm"):
        shutil.copy(os.path.join(rf.REF_DIR, f), dst)       # copies: FindBin::RealBin would follow a symlink back
    os.symlink(os.path.join(rf.REF_DIR, "rsem-build-read-index"), os.path.join(dst, "rsem-build-read-index"))
    src = rf.REF_DIR if which == "ref" else rf.BIN_DIR
    # ours: rsem-parse-alignments too - it writes the same text files plus the binary side-car rsem-run-em loads instead
    for tool in ("rsem-parse-alignments", "rsem-run-em", "rsem-run-gibbs"):
        os.symlink(os.path.join(src, tool), os.path.join(dst, tool))
    return dst


def _run(bindir, work, data, flags):
    os.makedirs(work)
    cmd = ["perl", os.path.join(bindir, "rsem-calculate-expression"), "--alignments", *flags, "--keep-intermediate-files",
           "--calc-pme", "--seed", "42", "-p", "2", os.path.join(data, "aln.sam"), os.path.join(data, "ref", "r"), "smp"]
    p = subprocess.run(cmd, cwd=work, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0, p.stdout[-3000:]
    return p.stdout


def _table(path):
    rows = [l.rstrip("\n").split("\t") for l in open(path)]
    return rows[0], rows[1:]


def _compare_tables(a, b):
    ha, ra = _table(a)
    hb, rb = _table(b)
    assert ha == hb and len(ra) == len(rb)
    for x, y in zip(ra, rb):
        for u, v in zip(x, y):
            try:
                fu, fv = float(u), float(v)
            except ValueError:
                assert u == v
                continue
            assert abs(fu - fv) <= 0.011 + 1e-6 * abs(fv), (x, y)


@pytest.fixture(scope="module")
def installs(tmp_path_factory, built):
    if not (rf.have_ref() and os.path.exists(DRIVER)):
        pytest.skip("oracle/_ref with the reference's Perl driver is not built here (oracle/Makefile builds it where the "
                    "reference sources are present)")
    if not shutil.which("perl"):
        pytest.skip("perl is not installed")
    base = tmp_path_factory.mktemp("acceptance")
    return base, _install(str(base / "bin_ref"), "ref"), _install(str(base / "bin_ours"), "ours")


CASES = {
    "se_noq": (0, ["--no-qualities"], dict(M=120, N1=4000, N0=200, read_len=50)),
    "pe_q": (3, ["--paired-end"], dict(M=150, N1=3000, N0=150, read_len=50, spurious=0.05)),
    "se_q_sampling": (1, ["--sampling-for-bam"], dict(M=100, N1=3000, N0=100, read_len=60)),
}


@pytest.mark.parametrize("name", list(CASES))
def test_perl_driver_with_our_binaries(installs, name):
    base, bin_ref, bin_ours = installs
    rt, flags, opts = CASES[name]
    data = rf.gen_dataset(str(base / f"{name}_data"), read_type=rt, sam=1, seed=21, **opts)
    out_ref = _run(bin_ref, str(base / f"{name}_ref"), data, flags)
    out_ours = _run(bin_ours, str(base / f"{name}_ours"), data, flags)
    assert " -b " in out_ref and " -b " in out_ours          # the default invocation asks for the posterior BAM
    wr, wo = str(base / f"{name}_ref"), str(base / f"{name}_ours")
    _compare_tables(f"{wo}/smp.isoforms.results", f"{wr}/smp.isoforms.results")
    _compare_tables(f"{wo}/smp.genes.results", f"{wr}/smp.genes.results")
    # the intermediate .dat the reference's parser wrote is what gen_dataset predicted (sid sign / strand coordinates)
    assert open(f"{wr}/smp.temp/smp.dat").read().split("\n", 1)[1] == open(f"{data}/s.temp/s.dat").read().split("\n", 1)[1]
    # our rsem-parse-alignments: the same text files, plus the side-car our rsem-run-em ran from
    for f in ("smp.dat", "smp.omit"):
        assert open(f"{wo}/smp.temp/{f}", "rb").read() == open(f"{wr}/smp.temp/{f}", "rb").read(), f
    assert open(f"{wo}/smp.stat/smp.cnt").read() == open(f"{wr}/smp.stat/smp.cnt").read()
    assert os.path.getsize(f"{wo}/smp.temp/smp.b200") > 0 and not os.path.exists(f"{wr}/smp.temp/smp.b200")
    tr, rr, ref = read_bam(f"{wr}/smp.transcript.bam")
    to, ro, ours = read_bam(f"{wo}/smp.transcript.bam")
    assert (tr, rr) == (to, ro) and len(ref) == len(ours) > 0
    n_zw = 0
    for a, b in zip(ours, ref):
        za, zb = a["tags"].pop("ZW", None), b["tags"].pop("ZW", None)
        assert (za is None) == (zb is None)
        if zb is not None:
            n_zw += 1
            assert za[0] == zb[0] == "f" and abs(za[1] - zb[1]) <= 1e-6 + 1e-6 * abs(zb[1])
            # MAPQ = round(-10 log10(1 - w)): equal unless w sits on a rounding boundary
            assert abs(a["mapq"] - b["mapq"]) <= (0 if abs(za[1] - zb[1]) == 0 else 1)
            a["mapq"] = b["mapq"]
        assert a == b
    assert n_zw > 0
    if "--sampling-for-bam" in flags:  # one alignment (or none: the noise entry) per read carries weight 1
        ws = np.array([r["tags"]["ZW"][1] if "ZW" in r["tags"] else -1 for r in read_bam(f"{wo}/smp.transcript.bam")[2]])
        assert set(np.unique(ws[ws >= 0])) <= {0.0, 1.0}
