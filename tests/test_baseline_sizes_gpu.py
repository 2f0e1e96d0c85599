"""Drop-in parity at the sizes BASELINE.json names (the small cases of test_dropin_gpu.py cannot catch a defect that only
shows with many tiles, long runs or the exit test):

  C1  configs[0], full size: 100 k single-end reads without qualities x 5 k transcripts, avg 5 hits -
      (a) 20 EM rounds against the reference (the "PR1 correctness" run), (b) FREE-RUNNING to convergence against the
      UNPATCHED reference binary: same exit ROUND (EM.cpp:416) and theta / TPM within 1e-6;
  C2  configs[1] at 1/5 scale (SURVEY.md section 6's probe): 2 M single-end reads with qualities x 50 k transcripts, 20 rounds;
  C3  configs[2] subsample: 1 M paired-end reads with qualities (2 x 100) against the full 200 k transcripts, 20 rounds.

Tolerance: 1e-6 relative on theta (>= 1e-7) and on the result rows' TPM (printed %.2f).  The reference's outputs are
stored in tests/golden/ref_outputs.json.gz (tools/make_golden_ref.py); at these sizes theta, the model and the result
rows are compared at a fixed seeded sample of ref_golden.KEEP positions each.
"""
import os
import re

import numpy as np
import pytest

import ref_golden
import rsem_files as rf

pytestmark = pytest.mark.gpu
THREADS = min(32, os.cpu_count() or 1)


@pytest.fixture(scope="module")
def workdir(tmp_path_factory, built):
    return tmp_path_factory.mktemp("baseline_sizes")


def _rounds(p):
    return [int(m.group(1)) for m in re.finditer(r"^ROUND = (\d+),", p.stdout, re.M)]


def _compare_outputs(g, ours):
    """our outputs in directory ours against the stored reference run g"""
    o = ref_golden.em_outputs(ours, ofg=False)
    raw_o, raw_r = g.take(o, "theta_raw"), g["theta_raw"]
    pol_o, pol_r = g.take(o, "theta_pol"), g["theta_pol"]
    assert rf.close_rel(raw_o, raw_r, 1e-6), rf.max_rel(raw_o, raw_r)
    assert rf.close_rel(pol_o, pol_r, 1e-6), rf.max_rel(pol_o, pol_r)
    mo, mr = g.take(o, "model"), g["model"]
    assert np.all(np.abs(mo - mr) <= 1e-9 + 1e-6 * np.abs(mr))
    for res in ("iso_res", "gene_res"):
        assert g.same(o, res + "_layout")
        xa, xb = g.take(o, res), g[res]
        assert np.all(np.abs(xa - xb) <= 0.011 + 1e-6 * np.abs(xb))
    return rf.max_rel(raw_o, raw_r)


@pytest.fixture(scope="module")
def c1_base(workdir):
    return rf.gen_dataset(str(workdir / "c1_base"), read_type=0, M=5000, N1=100_000, N0=5000, avg_family=5, read_len=50, seed=11)


def test_c1_full_size_20_rounds(workdir, c1_base):
    ours = rf.clone(c1_base, str(workdir / "c1_20_ours"))
    po = rf.run_em(ours, 0, "ours", rounds=20, gibbs_out=False)
    g = ref_golden.Run("baseline/c1_20")
    assert list(g["rounds"]) == _rounds(po) == list(range(1, 21))
    _compare_outputs(g, ours)


def test_c1_free_running_to_convergence(workdir, c1_base):
    """no round override on either side: MIN_ROUND 20, MAX_ROUND 10000, stop when no theta >= 1e-7 moves by >= 1e-3
    (EM.cpp:406-416); the stop test runs on the device in chunks of 32 rounds and must end on the reference's round"""
    ours = rf.clone(c1_base, str(workdir / "c1_free_ours"))
    po = rf.run_em(ours, 0, "ours", gibbs_out=False)
    g = ref_golden.Run("baseline/c1_free")     # the unpatched reference binary with -p 32
    exit_ref, ro = int(g["exit_round"][0]), _rounds(po)
    assert ro == list(range(1, len(ro) + 1)) and len(ro) > 20, "the data set is expected to need more than MIN_ROUND rounds"
    assert ro[-1] == exit_ref, f"exit round differs: ours {ro[-1]}, reference {exit_ref}"
    assert bool(g["max_round_warning"][0]) == ("Warning: RSEM reaches" in po.stderr)
    _compare_outputs(g, ours)


def test_c2_fifth_scale_20_rounds(workdir):
    base = rf.gen_dataset(str(workdir / "c2_base"), read_type=1, M=50_000, N1=2_000_000, N0=100_000, avg_family=10, read_len=100, seed=11)
    po = rf.run_em(base, 1, "ours", rounds=20, threads=THREADS, gibbs_out=False)
    g = ref_golden.Run("baseline/c2")
    assert list(g["rounds"]) == _rounds(po) == list(range(1, 21))
    _compare_outputs(g, base)


def test_c3_subsample_20_rounds(workdir):
    base = rf.gen_dataset(str(workdir / "c3_base"), read_type=3, M=200_000, N1=1_000_000, N0=50_000, avg_family=20, read_len=100, seed=11)
    po = rf.run_em(base, 3, "ours", rounds=20, threads=THREADS, gibbs_out=False)
    g = ref_golden.Run("baseline/c3")
    assert list(g["rounds"]) == _rounds(po) == list(range(1, 21))
    _compare_outputs(g, base)
