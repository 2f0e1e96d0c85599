#!/usr/bin/env python
"""Generate tests/golden/ref_outputs.json.gz and tests/golden/gibbs_in_*.tar.gz: what the reference binaries (oracle/_ref,
built by oracle/Makefile where the reference sources are present) write for the inputs of the parity tests in
test_parse_alignments.py, test_bam_io.py, test_sharding_multirank.py, test_dropin_gpu.py and test_baseline_sizes_gpu.py.  The tests compare
our executables against these stored outputs (tests/ref_golden.py describes the format).  Needs bin/ and tools/gen_dataset
(build()) and oracle/_ref; the C2 / C3 cases of test_baseline_sizes_gpu.py take several minutes of host time.

    python tools/make_golden_ref.py [group ...]     # groups: parse bam_io sharding dropin baseline (default: all)

A group named on the command line replaces that group's entries of ref_outputs.json.gz and keeps the others.
"""
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_golden as rg  # noqa: E402
import rsem_files as rf  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
GIBBS_INPUTS = ["s.temp/s.ofg", "s.stat/s.model", "s.temp/s.iso_res", "s.temp/s.gene_res"]


def _rounds(p):
    return np.array([int(m.group(1)) for m in re.finditer(r"^ROUND = (\d+),", p.stdout, re.M)], np.int64)


def _tree(out):
    import test_parse_alignments as tp
    files = tp._files(out)
    d = {"files": "\n".join(files)}
    for f in files:
        d["file:" + f] = rg.file_digest(os.path.join(out, f))
    return d


def group_parse(tmp):
    import test_parse_alignments as tp
    ref = os.path.join(rf.REF_DIR, "rsem-parse-alignments")
    out = {}
    for rt in (0, 1, 2, 3):
        d = rf.gen_dataset(f"{tmp}/b{rt}", read_type=rt, M=150, N1=3000, N0=200, read_len=50, var_len=30, seed=5 + rt,
                           sam=1, spurious=0.05, omit=7)
        assert tp._parse(ref, d, f"{d}/aln.sam", rt, f"{tmp}/b{rt}_sam").returncode == 0
        bam = f"{tmp}/b{rt}.bam"
        subprocess.check_call([tp.SELFTEST, "--bam-copy", f"{d}/aln.sam", bam, "2"], stdout=subprocess.DEVNULL)
        assert tp._parse(ref, d, bam, rt, f"{tmp}/b{rt}_bam").returncode == 0
        out[f"parse/byte_identical/{rt}/sam"] = rg.pack(_tree(f"{tmp}/b{rt}_sam"))
        out[f"parse/byte_identical/{rt}/bam"] = rg.pack(_tree(f"{tmp}/b{rt}_bam"))
    for rt in (1, 2):
        d = rf.gen_dataset(f"{tmp}/t{rt}", read_type=rt, M=80, N1=1500, N0=400, read_len=40, seed=3, sam=1)
        sam = tp._tag_some_unaligned(f"{d}/aln.sam", f"{tmp}/t{rt}.sam", rt >= 2)
        assert tp._parse(ref, d, sam, rt, f"{tmp}/t{rt}_out", ("-tag", "XM")).returncode == 0
        out[f"parse/tag/{rt}"] = rg.pack(_tree(f"{tmp}/t{rt}_out"))
    return out


def group_bam_io(tmp):
    d = rf.gen_dataset(f"{tmp}/d", read_type=3, M=30, N1=300, N0=20, read_len=40, sam=1, seed=9)
    rf.run_em(d, 3, "ref", rounds=2, threads=2, gibbs_out=False, extra=["-b", "aln.sam", "0"])
    return {"bam_io/htslib": rg.pack({"records": rg.bam_outputs(f"{d}/s.transcript.bam")["records"]})}


def group_sharding(tmp):
    out = {}
    for threads in (2, 3, 7):
        d = rf.gen_dataset(f"{tmp}/s{threads}", read_type=0, M=80, N1=900, N0=40, read_len=40, maxL=100, seed=threads)
        p = rf.run_em(d, 0, "ref", rounds=1, min_rounds=1, threads=threads, gibbs_out=False)
        split = np.array(re.findall(r"Thread \d+ : N = (\d+), NHit = (\d+)", p.stdout), np.int64).reshape(-1, 2)
        out[f"sharding/{threads}"] = rg.pack({"split": split.ravel()})
    return out


def _gibbs_base(tmp, tag, rt, seed, opts):
    """the reference's EM (12 rounds) on a generated data set; its outputs are the Gibbs sampler's inputs in the tests"""
    base = rf.gen_dataset(f"{tmp}/{tag}", read_type=rt, seed=seed, **opts)
    rf.run_em(base, rt, "ref", rounds=12, threads=1)
    # conprb to 6 significant digits (the archive is a third of the size); both samplers read this file
    with open(f"{base}/s.temp/s.ofg") as f:
        lines = f.read().split("\n")
    rounded = [lines[0]] + [" ".join(t if i % 2 == 0 else f"{float(t):.6g}" for i, t in enumerate(l.split())) for l in lines[1:]]
    with open(f"{base}/s.temp/s.ofg", "w") as f:
        f.write("\n".join(rounded))
    rg.write_tar(tag, base, GIBBS_INPUTS)
    return base


def group_dropin(tmp):
    import test_dropin_gpu as td
    out = {}
    for name, (rt, opts) in td.CASES.items():
        base = rf.gen_dataset(f"{tmp}/{name}", read_type=rt, seed=7, **opts)
        for rounds in (13, 3):
            d = rf.clone(base, f"{tmp}/{name}_{rounds}")
            p = rf.run_em(d, rt, "ref", rounds=rounds, threads=2)
            out[f"dropin/em/{name}/{rounds}"] = rg.pack(dict(rg.em_outputs(d), rounds=_rounds(p)))
    rt, opts = td.CASES["se_q_rspd_polyA"]
    base = _gibbs_base(tmp, "gibbs_in_se_q_rspd_polyA", rt, 3, dict(opts, omit=4))
    for threads, nsamples, gap in ((1, 7, 1), (3, 10, 2)):
        d = rf.clone(base, f"{tmp}/gibbs_{threads}")
        rf.run_gibbs(d, "ref", 15, nsamples, gap, threads, 12345)
        g = {f"countvectors{t}": rg.file_digest(f"{d}/s.temp/s.countvectors{t}") for t in range(threads)}
        g.update(rg.em_outputs(d, ofg=False, model=False, theta=False))
        out[f"dropin/gibbs/{threads}"] = rg.pack(g)
    rt, opts = td.CASES["se_noq"]
    base = _gibbs_base(tmp, "gibbs_in_se_noq", rt, 5, opts)
    td_prior = os.path.join(base, "prior.txt")
    with open(td_prior, "w") as f:
        rng = np.random.default_rng(0)
        for i in range(opts["M"]):
            f.write(f"{rng.uniform(0.1, 3.0):.4f} comment\n")
    for tag, extra in (("pc", ["--pseudo-count", "0.1"]), ("prior", ["--prior", "prior.txt"])):
        d = rf.clone(base, f"{tmp}/gibbs_{tag}")
        rf.run_gibbs(d, "ref", 10, 6, 1, 2, 99, extra=extra)
        g = {f"countvectors{t}": rg.file_digest(f"{d}/s.temp/s.countvectors{t}") for t in range(2)}
        g.update({k: v for k, v in rg.em_outputs(d, ofg=False, model=False, theta=False).items() if k.startswith("iso_res")})
        out[f"dropin/gibbs_{tag}"] = rg.pack(g)
    d = rf.gen_dataset(f"{tmp}/n1zero", read_type=0, M=30, N1=0, N0=50)
    subprocess.check_call([os.path.join(rf.REF_DIR, "rsem-run-em-rounds"), "ref/r", "0", "s", "s.temp/s", "s.stat/s"], cwd=d,
                          stdout=subprocess.DEVNULL)
    out["dropin/n1zero"] = rg.pack({r: rg.file_digest(f"{d}/s.temp/s.{r}") for r in ("iso_res", "gene_res")})
    for rt, sampling in ((3, False), (0, False), (1, True)):
        d = rf.gen_dataset(f"{tmp}/bam_{rt}", read_type=rt, M=80, N1=1500, N0=70, read_len=50, sam=1, seed=13 + rt)
        extra = ["-b", "aln.sam", "0"] + (["--sampling", "--seed", "4242"] if sampling else [])
        rf.run_em(d, rt, "ref", rounds=13, threads=2, gibbs_out=False, extra=extra)
        out[f"dropin/bam/{rt}"] = rg.pack(rg.bam_outputs(f"{d}/s.transcript.bam"))
    rt, opts = td.CASES["pe_q_rspd"]
    d = rf.gen_dataset(f"{tmp}/mgpu", read_type=rt, seed=9, **opts)
    rf.run_em(d, rt, "ref", rounds=14, threads=2)
    out["dropin/two_gpus"] = rg.pack(rg.em_outputs(d))
    return out


def group_baseline(tmp):
    out = {}
    cores = os.cpu_count() or 1
    c1_threads = 32     # test_baseline_sizes_gpu.py's -p on a machine with >= 32 cores
    c1 = rf.gen_dataset(f"{tmp}/c1", read_type=0, M=5000, N1=100_000, N0=5000, avg_family=5, read_len=50, seed=11)
    d = rf.clone(c1, f"{tmp}/c1_20")
    p = rf.run_em(d, 0, "ref", rounds=20, threads=c1_threads, gibbs_out=False)
    out["baseline/c1_20"] = rg.pack(dict(rg.em_outputs(d, ofg=False), rounds=_rounds(p)))
    d = rf.clone(c1, f"{tmp}/c1_free")
    p = rf.run_em(d, 0, "ref_unpatched", threads=c1_threads, gibbs_out=False)
    rounds = _rounds(p)
    out["baseline/c1_free"] = rg.pack(dict(rg.em_outputs(d, ofg=False), n_rounds=[len(rounds)], exit_round=rounds[-1:],
                                           max_round_warning=[int("Warning: RSEM reaches" in p.stderr)]))
    del c1
    for tag, rt, opts in (("c2", 1, dict(M=50_000, N1=2_000_000, N0=100_000, avg_family=10, read_len=100)),
                          ("c3", 3, dict(M=200_000, N1=1_000_000, N0=50_000, avg_family=20, read_len=100))):
        d = rf.gen_dataset(f"{tmp}/{tag}", read_type=rt, seed=11, **opts)
        p = rf.run_em(d, rt, "ref", rounds=20, threads=cores, gibbs_out=False)
        out[f"baseline/{tag}"] = rg.pack(dict(rg.em_outputs(d, ofg=False), rounds=_rounds(p)))
        shutil.rmtree(d)
    return out


GROUPS = {"parse": group_parse, "bam_io": group_bam_io, "sharding": group_sharding, "dropin": group_dropin, "baseline": group_baseline}


def main():
    if not rf.have_ref():
        sys.exit("oracle/_ref is missing: build it with `make -C oracle ref` where the reference sources are present")
    for g in sys.argv[1:] or list(GROUPS):
        with tempfile.TemporaryDirectory() as tmp:
            new = GROUPS[g](tmp)
        print(g, len(new), "runs", flush=True)
        runs = {k: v for k, v in (rg.load() if os.path.exists(rg.PATH) else {}).items() if not k.startswith(g + "/")}
        runs.update(new)
        rg.save(runs)
    print(rg.PATH, os.path.getsize(rg.PATH), "bytes")


if __name__ == "__main__":
    main()
