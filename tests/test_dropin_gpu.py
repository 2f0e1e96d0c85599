"""Drop-in parity: bin/rsem-run-em and bin/rsem-run-gibbs against the reference executables on the same generated inputs.
The reference's outputs (oracle/_ref, built from the reference sources by oracle/Makefile) are stored in
tests/golden/ref_outputs.json.gz, and the reference EM runs the Gibbs cases start from in tests/golden/gibbs_in_*.tar.gz
(tools/make_golden_ref.py); outputs longer than ref_golden.KEEP values are compared at a fixed seeded sample of positions.

Tolerances (north_star: theta / TPM within 1e-6 relative after the same iteration count; Gibbs: same
seed -> same draws):
  .theta (raw and polished)   1e-6 relative for theta >= 1e-7, 1e-12 absolute below
  .model tables (%.10g)       1e-6 relative / 1e-9 absolute
  .ofg conprb / ncpv          1e-6 relative
  result rows (%.2f)          0.011 absolute, or 1e-6 relative for large values
  .countvectors               byte-identical
"""
import filecmp
import os

import numpy as np
import pytest

import ref_golden
import rsem_files as rf

pytestmark = pytest.mark.gpu

CASES = {
    # name: (read_type, generator options)
    "se_noq": (0, dict(M=200, N1=3000, N0=150, read_len=50, maxL=200)),
    "se_q_rspd_polyA": (1, dict(M=150, N1=2500, N0=120, read_len=60, var_len=8, est_rspd=1, polyA=125, probF=0.7, spurious=0.05)),
    "pe_noq": (2, dict(M=150, N1=2000, N0=100, read_len=40, var_len=4, maxL=400, spurious=0.05)),
    "pe_q_rspd": (3, dict(M=200, N1=2500, N0=100, read_len=50, est_rspd=1, probF=0.3, spurious=0.1)),
    "se_q_revonly": (1, dict(M=100, N1=1500, N0=50, read_len=45, est_rspd=1, probF=0.0)),
    "se_noq_fraglen": (0, dict(M=100, N1=1500, N0=80, read_len=50, var_len=10, maxL=300, frag_mean=180, frag_sd=30)),
    "pe_q_polyA": (3, dict(M=120, N1=1500, N0=60, read_len=50, polyA=125, omit=5)),
}


def _res_close(g, o, res):
    """result rows: the same layout and text columns, numbers within 0.011 (printed %.2f) or 1e-6 relative"""
    assert g.same(o, res + "_layout")
    xa, xb = g.take(o, res), g[res]
    assert np.all(np.abs(xa - xb) <= 0.011 + 1e-6 * np.abs(xb)), float(np.max(np.abs(xa - xb)))


def _compare_em(g, o):
    """our rsem-run-em outputs o (ref_golden.em_outputs) against the stored reference run g"""
    raw_o, raw_r = g.take(o, "theta_raw"), g["theta_raw"]
    pol_o, pol_r = g.take(o, "theta_pol"), g["theta_pol"]
    assert rf.close_rel(raw_o, raw_r, 1e-6), rf.max_rel(raw_o, raw_r)
    assert rf.close_rel(pol_o, pol_r, 1e-6), rf.max_rel(pol_o, pol_r)
    mo, mr = g.take(o, "model"), g["model"]
    assert np.all(np.abs(mo - mr) <= 1e-9 + 1e-6 * np.abs(mr)), np.max(np.abs(mo - mr))
    assert g.same(o, "ofg_structure")      # M, N0, row pointers and transcript ids of the .ofg
    c_o, c_r = g.take(o, "ofg_conprb"), g["ofg_conprb"]
    assert np.all(np.abs(c_o - c_r) <= 1e-6 * np.abs(c_r))
    _res_close(g, o, "iso_res")
    _res_close(g, o, "gene_res")


@pytest.fixture(scope="module")
def workdir(tmp_path_factory, built):
    return tmp_path_factory.mktemp("dropin")


@pytest.mark.parametrize("rounds", [13, 3])
@pytest.mark.parametrize("name", list(CASES))
def test_em_matches_reference(workdir, name, rounds):
    rt, opts = CASES[name]
    base = rf.gen_dataset(str(workdir / f"{name}_base"), read_type=rt, seed=7, **opts)
    ours = rf.clone(base, str(workdir / f"{name}_{rounds}_ours"))
    po = rf.run_em(ours, rt, "ours", rounds=rounds)
    g = ref_golden.Run(f"dropin/em/{name}/{rounds}")     # the reference with -p 2
    # same number of rounds
    lo = [l for l in po.stdout.splitlines() if l.startswith("ROUND = ")]
    assert len(g["rounds"]) == len(lo) == rounds
    _compare_em(g, ref_golden.em_outputs(ours))


@pytest.mark.parametrize("threads,nsamples,gap", [(1, 7, 1), (3, 10, 2)])
def test_gibbs_same_seed_same_draws(workdir, threads, nsamples, gap):
    rt, opts = CASES["se_q_rspd_polyA"]
    base = rf.gen_dataset(str(workdir / f"gibbs_base_{threads}"), read_type=rt, seed=3, **dict(opts, omit=4))
    ref_golden.extract("gibbs_in_se_q_rspd_polyA", base)   # reference EM (12 rounds): .ofg (rounded) / .model / result rows
    ours = rf.clone(base, str(workdir / f"gibbs_ours_{threads}"))
    rf.run_gibbs(ours, "ours", 15, nsamples, gap, threads, 12345)
    g = ref_golden.Run(f"dropin/gibbs/{threads}")
    for t in range(threads):
        assert ref_golden.file_digest(f"{ours}/s.temp/s.countvectors{t}") == g[f"countvectors{t}"], f"countvectors{t} differ"
    o = ref_golden.em_outputs(ours, ofg=False, model=False, theta=False)
    _res_close(g, o, "iso_res")
    _res_close(g, o, "gene_res")


def test_gibbs_prior_and_pseudocount(workdir):
    rt, opts = CASES["se_noq"]
    base = rf.gen_dataset(str(workdir / "gibbs_prior_base"), read_type=rt, seed=5, **opts)
    ref_golden.extract("gibbs_in_se_noq", base)   # reference EM (12 rounds)
    M = opts["M"]
    with open(f"{base}/prior.txt", "w") as f:
        rng = np.random.default_rng(0)
        for i in range(M):
            f.write(f"{rng.uniform(0.1, 3.0):.4f} comment\n")
    for tag, extra in (("pc", ["--pseudo-count", "0.1"]), ("prior", ["--prior", "prior.txt"])):
        ours = rf.clone(base, str(workdir / f"gibbs_{tag}_ours"))
        rf.run_gibbs(ours, "ours", 10, 6, 1, 2, 99, extra=extra)
        g = ref_golden.Run(f"dropin/gibbs_{tag}")
        for t in range(2):
            assert ref_golden.file_digest(f"{ours}/s.temp/s.countvectors{t}") == g[f"countvectors{t}"], f"countvectors{t} differ"
        _res_close(g, ref_golden.em_outputs(ours, ofg=False, model=False, theta=False), "iso_res")


def test_no_alignable_reads(workdir):
    """N1 == 0 special case (EM.cpp:615-638): empty .theta / .model, zero result rows; no GPU work"""
    base = rf.gen_dataset(str(workdir / "n1zero_base"), read_type=0, M=30, N1=0, N0=50)
    ours = rf.clone(base, str(workdir / "n1zero_ours"))
    env_rounds = 3
    rf.run_em(ours, 0, "ours", rounds=env_rounds, gibbs_out=False)
    assert os.path.getsize(f"{ours}/s.stat/s.theta") == 0 and os.path.getsize(f"{ours}/s.stat/s.model") == 0
    g = ref_golden.Run("dropin/n1zero")     # the reference's result files, byte for byte
    assert ref_golden.file_digest(f"{ours}/s.temp/s.iso_res") == g["iso_res"]
    assert ref_golden.file_digest(f"{ours}/s.temp/s.gene_res") == g["gene_res"]


@pytest.mark.parametrize("rt,sampling", [(3, False), (0, False), (1, True)])
def test_posterior_bam(workdir, rt, sampling):
    """-b (EM.cpp:504-536, BamWriter.h): every alignment line of the input comes back with MAPQ and ZW:f from the posteriors;
    --sampling draws one alignment per read with the seeded MT19937 (sampling.h:50-65)"""
    base = rf.gen_dataset(str(workdir / f"bam_base_{rt}"), read_type=rt, M=80, N1=1500, N0=70, read_len=50, sam=1, seed=13 + rt)
    ours = rf.clone(base, str(workdir / f"bam_ours_{rt}"))
    extra = ["-b", "aln.sam", "0"] + (["--sampling", "--seed", "4242"] if sampling else [])
    po = rf.run_em(ours, rt, "ours", rounds=13, threads=3, gibbs_out=False, extra=extra)
    assert "Bam output file is generated!" in po.stdout
    g = ref_golden.Run(f"dropin/bam/{rt}")     # the reference with -p 2
    o = ref_golden.bam_outputs(f"{ours}/s.transcript.bam")
    # every field but ZW and MAPQ of every record (header included) is the reference's; ZW exactly on the mapped ones
    assert g.same(o, "records") and g.same(o, "has_zw")
    assert np.array_equal(np.isnan(o["zw"]), o["unmapped"])
    if sampling:
        assert set(np.unique(o["zw"][~o["unmapped"]])) <= {0.0, 1.0}
    zx, zy = g.take(o, "zw"), g["zw"]
    has = ~np.isnan(zy)
    assert np.all(np.abs(zx[has] - zy[has]) <= 1e-6 + 1e-6 * np.abs(zy[has]))
    # MAPQ = round(-10 log10(1 - w)): equal unless w sits on a rounding boundary
    same_w = (zx == zy) | ~has
    assert np.all(np.abs(g.take(o, "mapq") - g["mapq"]) <= np.where(same_w, 0, 1))


def test_bam_of_a_sample_without_alignable_reads(workdir):
    """N1 == 0 with -b: the input file is copied as it is (EM.cpp:627-633)"""
    base = rf.gen_dataset(str(workdir / "bam_n1zero"), read_type=0, M=30, N1=0, N0=50, sam=1)
    rf.run_em(base, 0, "ours", rounds=3, gibbs_out=False, extra=["-b", "aln.sam", "0"])
    assert filecmp.cmp(f"{base}/aln.sam", f"{base}/s.transcript.bam", shallow=False)


def test_em_two_gpus_matches_reference(workdir):
    """RSEM_B200_DEVICES=0,1: reads sharded over two GPUs (same rule as the reference's threads), counts and model
    statistics summed with ncclAllReduce inside the library.  Needs a machine with >= 2 GPUs."""
    import rsem_b200
    if rsem_b200.load_library().device_count() < 2:
        pytest.skip("needs two GPUs")
    rt, opts = CASES["pe_q_rspd"]
    base = rf.gen_dataset(str(workdir / "mgpu_base"), read_type=rt, seed=9, **opts)
    ours = rf.clone(base, str(workdir / "mgpu_ours"))
    os.environ["RSEM_B200_DEVICES"] = "0,1"
    try:
        po = rf.run_em(ours, rt, "ours", rounds=14)
    finally:
        del os.environ["RSEM_B200_DEVICES"]
    assert "GPU 1 : N = " in po.stdout
    _compare_em(ref_golden.Run("dropin/two_gpus"), ref_golden.em_outputs(ours))     # the reference with -p 2
