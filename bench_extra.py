"""bench.py --workload C4 (Gibbs sampler, BASELINE configs[3]) and --workload MODEL (one model-updating EM round).

Both go through the reference-facing boundary: C4 through the C ABI's gibbs_upload / gibbs_run with HOST buffers, MODEL
through the drop-in executable bin/rsem-run-em on generated intermediate files.  Same JSON contract as bench.py.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))


def _ofg_matrix(N, M, deg, seed):
    """the matrix rsem-run-em --gibbs-out hands to rsem-run-gibbs (Gibbs.cpp:119-131): per read the noise entry (sid 0)
    first, then its hits.  Transcripts form disjoint isoform families of 1 + Poisson(deg - 1) consecutive ids (genes);
    a read comes from one family (expression weights u^4: long tailed, as in tools/gen_dataset) and hits a run of its
    members - so the read x transcript graph falls into one connected component per family, as real data does per gene."""
    rng = np.random.default_rng(seed)
    sizes = []
    tot = 0
    while tot < M:
        k = min(int(1 + rng.poisson(deg - 1)), M - tot)
        sizes.append(k)
        tot += k
    sizes = np.array(sizes, np.int64)
    fam_start = np.concatenate([[1], 1 + np.cumsum(sizes)[:-1]])
    wgt = rng.random(len(sizes)) ** 4 + 1e-6
    fam = rng.choice(len(sizes), size=N, p=wgt / wgt.sum())
    fsz = sizes[fam]
    degs = np.maximum(1, np.minimum(fsz, np.where(rng.random(N) < 0.8, fsz, 1 + (rng.random(N) * fsz).astype(np.int64))))
    first = fam_start[fam] + ((fsz - degs) * rng.random(N)).astype(np.int64)
    w = degs + 1  # + noise entry
    row_ptr = np.zeros(N + 1, np.uint64)
    row_ptr[1:] = np.cumsum(w)
    E = int(row_ptr[-1])
    within = np.arange(E, dtype=np.int64) - np.repeat(row_ptr[:-1].astype(np.int64), w)
    sid = (np.repeat(first, w) + within - 1).astype(np.int32)
    sid[within == 0] = 0
    # conditional probabilities as the read models produce them: an alignment is a product of ~100 per-base match
    # probabilities times position / fragment-length priors (1e-12 .. 1e-3), the noise entry a product of ~100 background
    # base frequencies (~4^-100): a read leaves or joins the noise transcript only when its alignments are junk (2 % here)
    val = np.empty(E)
    CH = 20_000_000
    for a in range(0, E, CH):
        b = min(E, a + CH)
        val[a:b] = 10.0 ** rng.uniform(-12, -3, b - a)
    noise = 10.0 ** rng.uniform(-70, -50, N)
    junk = rng.random(N) < 0.02
    noise[junk] = 10.0 ** rng.uniform(-14, -6, int(junk.sum()))
    val[row_ptr[:-1].astype(np.int64)] = noise
    return row_ptr, sid, val, E


def run_gibbs(args):
    import torch  # noqa: F401  (device plumbing only: makes sure the CUDA context libraries are loaded the same way)

    import bench
    import rsem_b200
    from rsem_b200.capi import GibbsOut, GibbsParams

    N, M, deg = args.gibbs_reads, 50_000, 10
    chains = args.gibbs_chains
    t0 = time.perf_counter()
    row_ptr, sid, val, E = _ofg_matrix(N, M, deg, seed=2024)
    t_gen = time.perf_counter() - t0
    print(f"bench C4: matrix generated in {t_gen:.1f} s ({N} reads, {E} entries)", file=sys.stderr, flush=True)
    n0 = N / 20
    ctx = rsem_b200.Context(0)
    t0 = time.perf_counter()
    ctx.gibbs_upload(row_ptr, sid, val, M)
    t_upload = time.perf_counter() - t0
    print(f"bench C4: uploaded + components in {t_upload:.1f} s", file=sys.stderr, flush=True)

    init = np.zeros(M + 1, np.int32)
    alpha = np.ones(M + 1)
    totc = float(M + 1) + n0 + N
    rng = np.random.default_rng(1)
    eel = np.concatenate([[0.0], rng.uniform(200, 2000, M)])
    mw = np.ones(M + 1)
    genes = np.arange(1, M + 2, 4, dtype=np.int32)
    genes[-1] = M + 1
    seeds = (np.arange(chains, dtype=np.uint32) * np.uint32(2654435761) + np.uint32(12345)).astype(np.uint32)

    def run(burnin, per_chain):
        samples = np.full(chains, per_chain, np.int32)
        p = GibbsParams()
        p.M, p.burnin, p.gap, p.n_chains = M, burnin, 1, chains
        p.chain_samples = samples.ctypes.data_as(C.POINTER(C.c_int32))
        p.chain_seeds = seeds.ctypes.data_as(C.POINTER(C.c_uint32))
        p.n0, p.totc = n0, totc
        p.init_counts = init.ctypes.data_as(C.POINTER(C.c_int32))
        p.pseudo_counts = alpha.ctypes.data_as(C.POINTER(C.c_double))
        p.eel, p.mw = eel.ctypes.data_as(C.POINTER(C.c_double)), mw.ctypes.data_as(C.POINTER(C.c_double))
        p.n_genes = len(genes) - 1
        p.gene_start = genes.ctypes.data_as(C.POINTER(C.c_int32))
        cv = np.zeros((chains * per_chain, M + 1), np.int32)
        sums = [np.zeros(M + 1) for _ in range(4)] + [np.zeros(len(genes) - 1)]
        o = GibbsOut()
        o.count_vectors = cv.ctypes.data_as(C.POINTER(C.c_int32))
        o.sum_c, o.sum_c2, o.sum_tpm, o.sum_fpkm, o.sum_gene_c2 = (s.ctypes.data_as(C.POINTER(C.c_double)) for s in sums)
        t0 = time.perf_counter()
        ctx.gibbs_run(p, o)
        dt = time.perf_counter() - t0
        print(f"bench C4: gibbs_run burn-in {burnin}, {per_chain} samples per chain x {chains} chains: {dt:.2f} s", file=sys.stderr, flush=True)
        assert np.all(cv.sum(axis=1) == N + int(n0))  # every read is assigned to exactly one entry in every kept sample
        return dt, cv, sums

    run(2, 1)  # warm-up (allocations, first launch)
    W = max(args.warmup, 3)
    K = args.steps
    # W + 1 sweeps per chain, then W + 1 + K: the difference times exactly K sweeps (x chains) through the whole C-ABI call;
    # each twice, the faster one counts (allocation / first-touch noise of a call is of the order of 0.1 s)
    t_short = min(run(W, 1)[0], run(W, 1)[0])
    t_long1 = run(W, 1 + K)[0]
    t_long2, cv, sums = run(W, 1 + K)
    t_long = min(t_long1, t_long2)
    if args.dump_outputs:
        # all kept count vectors would be chains x (1 + K) x (M + 1) values: the last one of every chain is written
        last = cv.reshape(chains, 1 + K, M + 1)[:, -1, :]
        bench.dump_outputs(args.dump_outputs, last_count_vectors=last, sum_c=sums[0], sum_c2=sums[1], sum_tpm=sums[2],
                           sum_fpkm=sums[3], sum_gene_c2=sums[4])
    per_sweep_all = (t_long - t_short) / K          # one sweep of all chains, seconds
    chain_sweeps_per_s = chains / per_sweep_all
    # SURVEY.md 8(d): bytes per chain-sweep when C chains share the stream = (12 E + 8 N) / C + 8 N
    bytes_cs = (12 * E + 8 * N) / chains + 8 * N
    peak, peak_src = bench.measured_peak_gbs()
    achieved = bytes_cs * chains / per_sweep_all / 1e9
    full_job = t_long  # includes per-sample O(M) work and the D2H of the kept count vectors
    # CPU port on a bounded sample: one chain, first reads, a few sweeps
    cpu = None
    if not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_binding
        orc = oracle_binding.Oracle()
        ns = min(N, 1_000_000)
        es = int(row_ptr[ns])
        t0 = time.perf_counter()
        orc.gibbs_chain(row_ptr[: ns + 1].copy(), sid[:es].copy(), val[:es].copy(), M, ns / 20, init, alpha,
                        float(M + 1) + ns / 20 + ns, eel, mw, genes, 2, 1, 1, 777)
        dt = time.perf_counter() - t0
        cpu = {"value": 3 / dt * (es / E), "unit": "chain-sweeps/s (scaled to the full matrix)", "cores": 1, "kind": "port",
               "ns_per_entry_sweep": round(dt / 3 / es * 1e9, 3),
               "sample": f"oracle/librsem_oracle.so gibbs chain, first {ns} reads / {es} entries, 3 sweeps, 1 thread; the reference "
                         "runs one such chain per thread (Gibbs.cpp:207-254)"}
    out = {"metric": "gibbs_chain_sweeps_per_sec", "value": chain_sweeps_per_s, "unit": "chain-sweeps/s", "n_gpus": 1, "steps": K,
           "warmup": W, "ms_per_step": per_sweep_all * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64 weights, i32 counts, u32 MT19937 draws", "data": "synthetic",
           "config": {"workload": f"C4: Gibbs sampler, {N} reads x {M} transcripts, {E} .ofg entries (incl. {N} noise entries), "
                                  f"{chains} chains in lock-step (= rsem-run-gibbs -p {chains}); a step is one sweep of all chains",
                      "l2_policy": "inputs (1.3 GB) larger than L2, no flush needed"},
           "entries_per_sec": E * chain_sweeps_per_s,
           "e2e": {"value": chains * (W + 1 + K) / full_job, "unit": "chain-sweeps/s", "h2d_bytes_per_step": 0,
                   "d2h_bytes_per_step": chains * (M + 1) * 4,
                   "note": f"whole gibbs_run call ({W + 1 + K} sweeps per chain, {1 + K} kept samples per chain: per-sample theta / TPM "
                           "accumulation and the count vectors copied back to the host); the matrix was uploaded once: "
                           f"{t_upload:.1f} s incl. the host-side component analysis ({12 * E + 8 * N} B)"},
           "gpu_launches": ctx.launch_count(),
           "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                        "traffic": None, "kernel": "gibbs_parallel_kernel (K5)", "peak_source": peak_src,
                        "algorithmic_bytes_per_chain_sweep": bytes_cs,
                        "note": "SURVEY 8(d): (12 E + 8 N) / C + 8 N bytes per chain-sweep with C chains sharing the stream"},
           "cpu_baseline": cpu,
           "extrapolated": {"reference_job": "1000 samples, burn-in 200, gap 1 over 8 chains = 325 sweeps per chain",
                            "seconds": 325 * per_sweep_all * (8 / chains)},
           "host_seconds": {"generate": round(t_gen, 1), "upload_and_components": round(t_upload, 1)},
           "head": bench.git_head()}
    print(json.dumps(out), flush=True)
    ctx.close()


def run_model(args):
    """rounds 1-10 of rsem-run-em (EM.cpp:364-404): K1 (conprb) + K2 with posteriors + K3 (model statistics) per round,
    timed through the drop-in executable from its own ROUND lines; per-kernel times from RSEM_B200_PHASE_TIMING."""
    import bench

    gen = os.path.join(ROOT, "tools", "gen_dataset")
    exe = os.path.join(ROOT, "bin", "rsem-run-em")
    N, M, L = args.model_reads, 50_000, 100
    with tempfile.TemporaryDirectory(prefix="rsem_model_bench_") as d:
        t0 = time.perf_counter()
        subprocess.check_call([gen, "--out", d, "--read-type", "3", "--M", str(M), "--N1", str(N), "--N0", str(N // 20),
                               "--avg-family", "10", "--read-len", str(L), "--seed", "11"], stderr=subprocess.DEVNULL)
        t_gen = time.perf_counter() - t0
        with open(f"{d}/s.temp/s.dat") as f:
            H = int(f.readline().split()[1])
        rounds = 10 + max(args.warmup, 3)
        env = dict(os.environ, RSEM_MAX_ROUND=str(rounds), RSEM_MIN_ROUND=str(rounds), RSEM_B200_PHASE_TIMING="1")
        p = subprocess.Popen([exe, f"{d}/ref/r", "3", f"{d}/s", f"{d}/s.temp/s", f"{d}/s.stat/s", "-p", str(min(32, os.cpu_count() or 1))],
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env, text=True, bufsize=1)
        stamps = {}
        t_start = time.perf_counter()
        for line in p.stdout:
            if line.startswith("ROUND = "):
                stamps[int(line.split(",")[0].split("=")[1])] = time.perf_counter()
        err = p.stderr.read()
        rc = p.wait()
        wall = time.perf_counter() - t_start
    if rc != 0:
        print(json.dumps({"metric": "model_round_hits_per_sec", "error": err[-400:]}))
        return
    per_round = (stamps[2 + args.steps] - stamps[2]) / args.steps   # rounds 3..10 (rounds 1-2 carry the first launches)
    phases = [l for l in err.splitlines() if "phase timing" in l]
    # SURVEY 8(d) "K1/K3 rounds": per read its bases + qualities once per kernel, per hit 2 L reference bases + hit fields
    k1 = N * 4 * L + H * (2 * L + 4 + 4 + 4 + 8)
    k3 = N * 4 * L + H * (2 * L + 4 + 4 + 4 + 8)
    k2 = 12 * H + 16 * N + 8 * H + 8 * N
    peak, peak_src = bench.measured_peak_gbs()
    out = {"metric": "model_round_hits_per_sec", "value": H / per_round, "unit": "hits/s", "n_gpus": 1, "steps": args.steps, "warmup": 2,
           "ms_per_step": per_round * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic",
           "config": {"workload": f"MODEL: one model-updating EM round (K1 conprb + K2 with posteriors + K3 statistics + host "
                                  f"Model::finish), PairedEndQModel, {N} reads 2 x {L}, {M} transcripts, {H} hits, through bin/rsem-run-em"},
           "reads_per_sec": N / per_round,
           "e2e": {"value": H / per_round, "unit": "hits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "note": f"whole executable {wall:.1f} s for {rounds} rounds incl. parsing and the final pass"},
           "roofline": {"bound": "hbm", "achieved": round((k1 + k2 + k3) / per_round / 1e9, 1), "peak": peak, "unit": "GB/s",
                        "frac": round((k1 + k2 + k3) / per_round / 1e9 / peak, 4), "traffic": None, "peak_source": peak_src,
                        "kernel": "conprb_kernel + estep (posteriors) + update_q_kernel",
                        "algorithmic_bytes": {"K1": k1, "K2_post": k2, "K3": k3},
                        "note": "latency / table-lookup bound kernels: the fraction is reported, the 60 % target applies to K2 only"},
           "phase_timing": phases, "host_seconds": {"generate": round(t_gen, 1)}, "gpu_launches": None,
           "cpu_baseline": None, "head": bench.git_head()}
    print(json.dumps(out), flush=True)
