#!/usr/bin/env python
"""bench.py - throughput of librsem_b200's EM / Gibbs hot path on B200, and the reference's CPU arm.

Metric (BASELINE.json): EM reads*hits/s (= hits streamed per second by the frozen-conprb E+M round, rounds >= 12 of the
reference's EM loop) and the equivalent EM iterations/s; HBM GB/s against the roofline.

  python bench.py                                        # workload C3 (BASELINE configs[2]) on one GPU
  torchrun ... bench.py --gpus N [--scaling strong]      # weak: one C3 shard per GPU; strong: ONE C3 matrix sharded by
                                                         # the reference's rule (EM.cpp:135-157) over N GPUs
  python bench.py --workload C1|C2|C5                    # the other EM configs (C5 = Zipf degrees <= 200)
  python bench.py --workload C4                          # Gibbs sampler (BASELINE configs[3]): chain-sweeps/s
  python bench.py --workload MODEL                       # one model round (K1 + K2 with posteriors + K3), rounds 1-10
  python bench.py --impl reference                       # oracle/_ref/rsem-run-em (the unmodified reference) on the host cores
  python bench.py --dump-outputs DIR                     # also write what the last timed step returned to DIR/*.npy
                                                         # (float64), to compare two builds (EM workloads and C4)

A "step" is one EM round = K2 (E-step + count accumulation) [+ NCCL allreduce of the count vector when N > 1] + K4 (theta
update, convergence test) over the resident hit matrix.  The matrix (>= 9 GB at C3) is far larger than L2 (126 MB), so
no explicit L2 flush is needed; C1 fits L2 and says so.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (reads, transcripts, mean hits/read, zipf)            BASELINE.json configs[0..2], [4]
    "C1": (100_000, 5_000, 5, False),
    "C2": (10_000_000, 50_000, 10, False),
    "C3": (50_000_000, 200_000, 20, False),
    "C5": (50_000_000, 200_000, 0, True),
}
E2E_ROUNDS = (100, 20)  # frozen-conprb rounds per end-to-end job (the reference runs >= 20, typically 100s-1000s)
BIG = 1 << 30


def alg_bytes(N, H, M):
    """SURVEY.md section 8(d): 12 B per hit + 16 B per read + 16 B per transcript"""
    return 12 * H + 16 * N + 16 * (M + 1)


# --------------------------------------------------------------------------------------------------
def gen_degrees(torch, dev, N, M, deg, seed, zipf=False):
    """degree of every read: 1 + Poisson(deg - 1), or Zipf(1.1) truncated at 200 (C5: the aligner caps RSEM passes,
    rsem-calculate-expression:40,83,408,442)"""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    if zipf:
        k = torch.arange(1, 201, device=dev, dtype=torch.float64)
        p = k.pow(-1.1)
        degs = torch.empty(N, dtype=torch.int64, device=dev)
        for a in range(0, N, 10_000_000):
            b = min(N, a + 10_000_000)
            degs[a:b] = torch.multinomial(p, b - a, replacement=True, generator=g) + 1
    else:
        degs = 1 + torch.poisson(torch.full((N,), float(deg - 1), device=dev), generator=g).to(torch.int64)
    degs.clamp_(max=min(M, 1000))
    return degs


def gen_rows(torch, dev, degs, M, seed):
    """rows with the given degrees: a row hits consecutive transcript ids (isoform families are contiguous) from a
    random start, conprb ~ 10^U(-60,-3), ncpv ~ 10^U(-80,-40)  (SURVEY.md section 8(d))"""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    N = degs.numel()
    row_ptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    torch.cumsum(degs, 0, out=row_ptr[1:])
    H = int(row_ptr[-1].item())
    start = torch.randint(1, M + 1, (N,), device=dev, generator=g, dtype=torch.int64)
    start = torch.minimum(start, M - degs + 1).clamp_(min=1)
    sid = torch.empty(H, dtype=torch.int32, device=dev)
    CH = 5_000_000  # rows per chunk: bounds the int64 temporaries
    for a in range(0, N, CH):
        b = min(N, a + CH)
        ha, hb = int(row_ptr[a].item()), int(row_ptr[b].item())
        rows = torch.repeat_interleave(torch.arange(a, b, device=dev), degs[a:b])
        within = torch.arange(ha, hb, device=dev) - row_ptr[rows]
        s = (start[rows] + within).to(torch.int32)
        sign = torch.randint(0, 2, (hb - ha,), device=dev, generator=g, dtype=torch.int32) * 2 - 1
        sid[ha:hb] = s * sign
        del rows, within, s, sign
    conprb = torch.empty(H, dtype=torch.float64, device=dev)
    for a in range(0, H, 100_000_000):
        b = min(H, a + 100_000_000)
        u = torch.rand(b - a, device=dev, generator=g, dtype=torch.float64)
        conprb[a:b] = torch.pow(10.0, -60.0 + 57.0 * u)
        del u
    ncpv = torch.pow(10.0, -80.0 + 40.0 * torch.rand(N, device=dev, generator=g, dtype=torch.float64))
    return row_ptr, sid, conprb, ncpv, H


def gen_matrix_torch(torch, dev, N, M, deg, seed, zipf=False):
    degs = gen_degrees(torch, dev, N, M, deg, seed, zipf)
    return gen_rows(torch, dev, degs, M, seed + 7)


def small_matrix_numpy(N, M, deg, seed):
    """seeded host matrix for the multi-rank parity check (same on every rank)"""
    rng = np.random.default_rng(seed)
    degs = np.minimum(1 + rng.poisson(deg - 1, N), M)
    row_ptr = np.zeros(N + 1, np.uint64)
    row_ptr[1:] = np.cumsum(degs)
    H = int(row_ptr[-1])
    start = np.minimum(rng.integers(1, M + 1, N), M - degs + 1).clip(1)
    sid = (np.repeat(start, degs) + (np.arange(H) - np.repeat(row_ptr[:-1].astype(np.int64), degs))).astype(np.int32)
    sid *= np.where(rng.random(H) < 0.5, 1, -1).astype(np.int32)
    return row_ptr, sid, 10.0 ** rng.uniform(-60, -3, H), 10.0 ** rng.uniform(-80, -40, N)


class ClockSampler:
    """nvidia-smi sampling while the GPU runs the timed workload (B200_PROFILING.md 'clocks' recipe).
    nvidia-smi needs ~0.2 s to start and samples every 100 ms, so it is started before the warm-up and only
    samples whose time stamp lies inside [t0, t1] (GPU under the benchmark's load) are used."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.p, self.f = index, None, None

    def start(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def _rows(self):
        out = []
        try:
            with open(self.f.name) as f:
                for line in f:
                    c = [x.strip() for x in line.split(",")]
                    if len(c) < 10:
                        continue
                    try:
                        ts = time.mktime(time.strptime(c[0].split(".")[0], "%Y/%m/%d %H:%M:%S")) + float("0." + c[0].split(".")[1])
                        out.append((ts, float(c[2]), float(c[3]), c[6:10]))
                    except (ValueError, IndexError):
                        continue
        except Exception:
            pass
        return out

    def wait_first(self, timeout=3.0):
        t = time.time()
        while self.p and time.time() - t < timeout and not self._rows():
            time.sleep(0.05)

    def count_since(self, t0):
        return sum(1 for r in self._rows() if r[0] >= t0)

    def stop(self, t0, t1):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r for r in self._rows() if t0 <= r[0] <= t1 + 0.05]
        os.unlink(self.f.name)
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm = [r[1] for r in rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[2] for r in rows) if rows else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "timed region + identical rounds right after it (nvidia-smi -lms 100)"}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def git_head():
    try:
        return subprocess.check_output(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], text=True, stderr=subprocess.DEVNULL).strip()
    except Exception:
        return None


# --------------------------------------------------------------------------------------------------
def cpu_baseline(oracle_mod, row_ptr, sid, conprb, ncpv, M, n0, budget_s=12.0):
    """the oracle port (OpenMP, all host cores, threads pinned through OMP_PROC_BIND / OMP_PLACES set in main()) on a
    bounded sample of the same workload: 3 repeats, the median is reported and the spread kept"""
    orc = oracle_mod.Oracle()
    cores = os.cpu_count() or 1
    N = len(row_ptr) - 1
    theta = np.empty(M + 1)
    theta[0] = max(n0 / (N + n0), 1e-8)
    theta[1:] = (1 - theta[0]) / M
    H = int(row_ptr[-1])
    t0 = time.perf_counter()
    theta, _, _ = orc.em_rounds(row_ptr, sid, conprb, ncpv, theta, n0, 12, 2, BIG, BIG, n_threads=cores)
    per = (time.perf_counter() - t0) / 2
    rounds = int(max(3, min(100, budget_s / 3 / max(per, 1e-4))))
    vals = []
    for _ in range(3):
        t0 = time.perf_counter()
        orc.em_rounds(row_ptr, sid, conprb, ncpv, theta, n0, 14, rounds, BIG, BIG, n_threads=cores)
        vals.append(H * rounds / (time.perf_counter() - t0))
    return {"value": float(np.median(vals)), "unit": "hits/s", "cores": cores, "kind": "port",
            "repeats_hits_per_s": [float(f"{v:.4g}") for v in vals],
            "sample": f"first {N} reads / {H} hits of the workload matrix, 3 x {rounds} frozen-conprb rounds (median), "
                      f"oracle/librsem_oracle.so with {cores} OpenMP threads (OMP_PROC_BIND=spread, OMP_PLACES=cores)"}


def multi_rank_parity(torch, dist, rsem_b200, local, world, rank, uid):
    """ONE seeded small matrix, sharded by the library's rule (the reference's, EM.cpp:135-157): 5 rounds over the NCCL path
    must give the theta of a single-GPU run of the whole matrix, and the same theta on every rank."""
    N, M = 200_000, 5_000
    row_ptr, sid, conprb, ncpv = small_matrix_numpy(N, M, 8, seed=4242)
    n0 = N / 20
    theta0 = np.empty(M + 1)
    theta0[0] = max(n0 / (N + n0), 1e-8)
    theta0[1:] = (1 - theta0[0]) / M
    lib = rsem_b200.load_library()
    a, b = lib.shard_reads(row_ptr, world)[rank]
    h0, h1 = int(row_ptr[a]), int(row_ptr[b])
    ctx = rsem_b200.Context(local)
    ctx.comm_init(uid, world, rank)
    ctx.upload_hits((row_ptr[a:b + 1] - np.uint64(h0)).astype(np.uint64), sid[h0:h1], M)
    ctx.upload_conprb(conprb[h0:h1], ncpv[a:b])
    ctx.set_theta(theta0)
    ctx.em_rounds(12, 5, BIG, BIG, n0)
    th = ctx.get_theta()
    ctx.close()
    dev = torch.device("cuda", local)
    mine = torch.from_numpy(th).to(dev)
    allth = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allth, mine)
    identical = all(bool(torch.equal(allth[0], t)) for t in allth)
    err = None
    if rank == 0:
        ctx = rsem_b200.Context(local)
        ctx.upload_hits(row_ptr, sid, M)
        ctx.upload_conprb(conprb, ncpv)
        ctx.set_theta(theta0)
        ctx.em_rounds(12, 5, BIG, BIG, n0)
        ref = ctx.get_theta()
        ctx.close()
        big = ref >= 1e-7
        err = float(np.max(np.abs(th[big] - ref[big]) / ref[big]))
        shards = [(y - x, int(row_ptr[y] - row_ptr[x])) for x, y in lib.shard_reads(row_ptr, world)]
        print(f"bench: multi-rank parity: {world} ranks, shards (reads, hits) {shards}, 5 rounds, theta identical on all "
              f"ranks: {identical}, max rel err vs single-GPU run: {err:.2e}", file=sys.stderr, flush=True)
        assert identical and err <= 1e-12, "multi-rank EM differs from the single-GPU run"
    return {"reads": N, "rounds": 5, "ranks_identical": identical, "max_rel_err_vs_single_gpu": err}


def measure_traffic(args, name):
    """dram bytes per K2 launch, measured now: the same workload in a child process under ncu (one launch)"""
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none",
           "-k", "regex:estep_class_kernel|estep_rows_kernel|estep_direct_kernel", "-s", "3", "-c", "1", "--csv",
           sys.executable, os.path.abspath(__file__), "--traffic-probe", "--workload", name, "--scale", str(args.scale)]
    if args.deg:
        cmd += ["--deg", str(args.deg)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600).stdout
    except Exception as e:
        return None, f"ncu failed: {e}"
    scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    rd = wr = kern = None
    for line in out.splitlines():
        c = [x.strip('"') for x in line.strip().split('","')]
        if len(c) < 5:
            continue
        try:
            if "dram__bytes_read.sum" in line:
                rd, kern = float(c[-1].replace(",", "")) * scale[c[-2]], c[4]
            if "dram__bytes_write.sum" in line:
                wr = float(c[-1].replace(",", "")) * scale[c[-2]]
        except (ValueError, KeyError):
            continue
    if rd is None or wr is None:
        return None, "ncu output not understood"
    return rd + wr, f"ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch of {kern.split('(')[0][-48:]}, measured in this run"


# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import rsem_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    name = args.workload
    N_full, M, deg, zipf = WORKLOADS[name]
    if args.scale != 1.0:
        N_full = max(1000, int(N_full * args.scale))
    if args.deg:
        deg = args.deg
    strong = args.scaling == "strong" and world > 1

    ctx = rsem_b200.Context(local)
    stream = torch.cuda.Stream(device=dev)
    ctx.set_stream(stream.cuda_stream)
    parity = None
    if world > 1:
        uid = [ctx.lib.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], world, rank)
        uid2 = [ctx.lib.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid2, src=0)
        parity = multi_rank_parity(torch, dist, rsem_b200, local, world, rank, uid2[0])

    if strong:
        # ONE matrix of N_full reads: every rank draws the same degrees, the library's rule cuts it, a rank fills its rows
        degs = gen_degrees(torch, dev, N_full, M, deg, 1234, zipf)
        rp_host = np.zeros(N_full + 1, np.uint64)
        rp_host[1:] = torch.cumsum(degs, 0).cpu().numpy().astype(np.uint64)
        a, b = ctx.lib.shard_reads(rp_host, world)[rank]
        total_hits = int(rp_host[-1])
        del rp_host
        row_ptr, sid, conprb, ncpv, H = gen_rows(torch, dev, degs[a:b].clone(), M, 1234 + 7 + 1000 * rank)
        del degs
        N = b - a
        n0 = N_full / 20
    else:
        N = N_full
        row_ptr, sid, conprb, ncpv, H = gen_matrix_torch(torch, dev, N, M, deg, 1234 + rank, zipf)
        total_hits = H * world  # every rank holds an equally shaped shard (weak scaling)
        n0 = N * world / 20
    if args.sort_rows:
        row_ptr, sid, conprb, ncpv = sort_rows_torch(torch, row_ptr, sid, conprb, ncpv, args.sort_rows)
    # the generator ran on torch's default stream, the context copies on its own (non-blocking) stream: the tensors
    # must be complete before they are adopted
    torch.cuda.synchronize()
    ctx.adopt_device_matrix(N, H, M, row_ptr.data_ptr(), sid.data_ptr(), conprb.data_ptr(), ncpv.data_ptr())
    if args.variant:
        ctx.set_estep_variant(args.variant)
    n_tot = (N_full if strong else N * world)
    theta0 = np.empty(M + 1)
    theta0[0] = max(n0 / (n_tot + n0), 1e-8)
    theta0[1:] = (1 - theta0[0]) / M
    ctx.set_theta(theta0)

    if args.traffic_probe:  # child of measure_traffic(): a few rounds for ncu to pick a launch from
        ctx.em_rounds(12, 6, BIG, BIG, n0)
        ctx.close()
        return

    # host copies for the e2e leg and the CPU baseline sample (before the device tensors are dropped)
    e2e_host = None
    sample = None
    e2e_err = "skipped (--no-e2e)"
    if not args.no_e2e:
        try:
            e2e_host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in (row_ptr, sid, conprb, ncpv)]
            for h, t in zip(e2e_host, (row_ptr, sid, conprb, ncpv)):
                h.copy_(t)
        except Exception as e:  # not enough host memory for the pinned copy
            e2e_host = None
            e2e_err = str(e).splitlines()[0]
    if rank == 0 and not args.no_cpu_baseline:
        ns = min(N, 2_000_000)
        hs = int(row_ptr[ns].item())
        sample = (row_ptr[: ns + 1].cpu().numpy().astype(np.uint64), sid[:hs].cpu().numpy(), conprb[:hs].cpu().numpy(),
                  ncpv[:ns].cpu().numpy())
    del row_ptr, sid, conprb, ncpv
    torch.cuda.empty_cache()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up + timed region (device-resident inputs) ------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first()
    ctx.em_rounds(12, args.warmup, BIG, BIG, n0)  # builds the class layout on the first round (not timed here, timed in e2e)
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_load0 = time.time()
    with torch.cuda.stream(stream):
        e0.record(stream)
        stats, _ = ctx.em_rounds(12 + args.warmup, args.steps, BIG, BIG, n0)
        e1.record(stream)
    barrier()
    launches = ctx.launch_count() - l0
    cta_ns = ctx.estep_cta_times().astype(np.float64)
    if args.dump_outputs and rank == 0:
        # what em_rounds hands its caller after the last timed step: theta and that round's (sum, bchange, totnum)
        dump_outputs(args.dump_outputs, theta=ctx.get_theta(), round_stats=np.array(stats[-1], np.float64))
    # keep the same load running until nvidia-smi has a few samples of it (a 20-round region lasts 50 ms)
    extra = 0
    while world == 1 and sampler.count_since(t_load0) < 5 and time.time() - t_load0 < 2.5:
        ctx.em_rounds(12 + args.warmup + args.steps + extra, 20, BIG, BIG, n0)
        extra += 20
    if world > 1:  # every rank must take part in the allreduce of each round: a fixed continuation
        ctx.em_rounds(12 + args.warmup + args.steps, 200, BIG, BIG, n0)
    t_load1 = time.time()
    clocks = sampler.stop(t_load0, t_load1) if rank == 0 else None
    ms_local = e0.elapsed_time(e1)
    ms = ms_local
    per_rank_ms = [ms_local / args.steps]
    if world > 1:
        t = torch.tensor([ms_local], device=dev, dtype=torch.float64)
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank_ms = [float(x.item()) / args.steps for x in allt]
        ms = max(float(x.item()) for x in allt)
    assert len(stats) == args.steps
    ms_per_step = ms / args.steps
    value = total_hits / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel (K2), per-launch CUDA events on the launching stream ------
    ctx.set_profiling(True)
    ctx.estep_timing(reset=True)
    ctx.em_rounds(12 + args.warmup + args.steps, max(3, min(10, args.steps)), BIG, BIG, n0)
    ctx.sync()
    k2_ms, k2_n = ctx.estep_timing(reset=True)
    ctx.set_profiling(False)
    peak, peak_src = measured_peak_gbs()
    ab = alg_bytes(N, H, M)
    cls = ctx.class_layout_info()
    k2_s = k2_ms / k2_n * 1e-3
    achieved = ab / k2_s / 1e9
    kernel = "estep_class_kernel (K2 on the equivalence-class layout)" if cls["built"] else "estep_rows_kernel (K2 on the CSR stream)"
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": None, "kernel": kernel,
                "algorithmic_bytes_per_launch": ab, "k2_ms_per_launch": round(k2_ms / k2_n, 4), "peak_source": peak_src,
                "note": "achieved = SURVEY 8(d) bytes (12 H + 16 N + 16 (M + 1)) / K2 time; the class layout stores ids once per "
                        "segment and no row pointers, so the bytes it actually streams are fewer (streamed_*)"}
    if cls["built"]:
        streamed = cls["bytes_per_round"] + 16 * (M + 1)
        roofline["streamed_bytes_per_launch"] = streamed
        roofline["streamed_gbs"] = round(streamed / k2_s / 1e9, 1)
        roofline["streamed_frac_of_peak"] = round(streamed / k2_s / 1e9 / peak, 4)
    if rank == 0 and world == 1 and not args.no_traffic:
        roofline["traffic"], roofline["traffic_source"] = measure_traffic(args, name)
    balance = None
    if cta_ns.size:
        balance = {"ctas": int(cta_ns.size), "cta_busy_us_min": round(float(cta_ns.min()) / 1e3, 1),
                   "cta_busy_us_median": round(float(np.median(cta_ns)) / 1e3, 1),
                   "cta_busy_us_max": round(float(cta_ns.max()) / 1e3, 1),
                   "max_over_mean": round(float(cta_ns.max() / cta_ns.mean()), 4),
                   "note": "busy time of the persistent K2 CTAs (one per SM) in the last timed launch, rank 0"}

    # ---- end to end through the C ABI with HOST buffers --------------------------------------------
    e2e = None
    if e2e_host is not None:
        hr, hsid, hc, hn = e2e_host
        bytes_in = hr.numel() * 8 + hsid.numel() * 4 + hc.numel() * 8 + hn.numel() * 8 + (M + 1) * 8
        bytes_out = (M + 1) * 8

        phases = {}

        def job(rounds):
            t = [time.perf_counter()]
            ctx.upload_hits_ptr(N, H, M, hr.data_ptr(), hsid.data_ptr())
            t.append(time.perf_counter())
            ctx.upload_conprb_ptr(hc.data_ptr(), hn.data_ptr())
            t.append(time.perf_counter())
            ctx.set_theta(theta0)
            ctx.em_rounds(12, rounds, BIG, BIG, n0)
            t.append(time.perf_counter())
            th = ctx.get_theta()
            t.append(time.perf_counter())
            phases.setdefault(rounds, []).append({"upload_hits": round(t[1] - t[0], 4), "upload_conprb": round(t[2] - t[1], 4),
                                                  "rounds": round(t[3] - t[2], 4), "get_theta": round(t[4] - t[3], 4)})
            return th

        res = {}
        for rounds in E2E_ROUNDS:
            job(rounds)  # warm-up
            barrier()
            n_jobs = 3
            times = []
            for _ in range(n_jobs):
                t0 = time.perf_counter()
                th = job(rounds)
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t0)
            if world > 1:   # a job ends when its slowest rank does
                t = torch.tensor(times, device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                times = [float(x) for x in t.tolist()]
            assert abs(th.sum() - 1.0) < 1e-9
            dt = sorted(times)[len(times) // 2]   # median job: about one upload_hits in four takes 3-5x longer (cause not identified), see profiles/README.md
            res[rounds] = (total_hits * rounds / dt, dt, [round(x, 4) for x in times])
        r0 = E2E_ROUNDS[0]
        e2e = {"value": res[r0][0], "unit": "hits/s", "h2d_bytes_per_step": bytes_in // r0, "d2h_bytes_per_step": bytes_out // r0,
               "h2d_bytes_per_job": bytes_in, "d2h_bytes_per_job": bytes_out, "rounds_per_job": r0, "jobs": 3,
               "seconds_per_job": round(res[r0][1], 4), "seconds_of_each_job": res[r0][2], "statistic": "median job",
               "phases_s_per_job": phases[r0][1:],
               "note": "job = upload CSR (row_ptr, sid) from pinned host memory + tiles (upload_hits), upload conprb / ncpv while "
                       "the class directory is built on the device (upload_conprb), gather the value stream and run the rounds, read "
                       "theta back; phases of the timed jobs (the warm-up job is left out); a step is one round, so the per-step "
                       "bytes are the job's bytes / rounds_per_job"}
        for rounds in E2E_ROUNDS[1:]:
            e2e[f"value_at_{rounds}_rounds_per_job"] = res[rounds][0]
            e2e[f"seconds_per_job_at_{rounds}_rounds"] = round(res[rounds][1], 4)
    else:
        e2e = {"value": None, "unit": "hits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
               "note": "no end-to-end leg: " + e2e_err}

    cpu = None
    if rank == 0 and sample is not None:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_binding
        cpu = cpu_baseline(oracle_binding, *sample, M, len(sample[3]) / 20)

    if rank == 0:
        shape = "Zipf(1.1) degrees <= 200" if zipf else f"mean degree {H / N:.2f}"
        out = {
            "metric": "em_reads_hits_per_sec", "value": value, "unit": "hits/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "em_iterations_per_sec": 1e3 / ms_per_step,
            "config": {"workload": f"{name}: {N_full} reads x {M} transcripts, {total_hits if strong else H} hits "
                                   f"{'in total' if strong else 'per GPU'} ({shape}), frozen-conprb E+M round (EM.cpp rounds >= 12)",
                       "reads_per_gpu": N, "transcripts": M, "hits_per_gpu": H, "total_hits": total_hits,
                       "l2_policy": "inputs (>= 9 GB) larger than L2, no flush needed" if H * 8 > 2e8 else "inputs fit L2 (launch-bound config)",
                       "parallelism": (f"{'ONE matrix' if strong else 'one shard per GPU'}, reads sharded over {world} GPUs by the "
                                       "reference's rule, ncclAllReduce(count) per round") if world > 1 else "1 GPU"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "class_layout": cls, "load_balance": balance, "per_rank_ms_per_step": [round(x, 4) for x in per_rank_ms],
            "multi_rank_parity": parity, "head": git_head(),
        }
        print(json.dumps(out), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(d, **arrays):
    """writes each array as DIR/<name>.npy in float64; the inputs of every workload are seeded, so two builds run with the
    same arguments can be compared file by file"""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, f"{name}.npy"), np.ascontiguousarray(a, np.float64))


def sort_rows_torch(torch, row_ptr, sid, conprb, ncpv, by):
    """Experiment: rows reordered by their first transcript id or by their degree."""
    N = row_ptr.numel() - 1
    degs = row_ptr[1:] - row_ptr[:-1]
    key = sid[row_ptr[:-1]].abs() if by == "start" else degs
    perm = torch.argsort(key, stable=True)
    nd = degs[perm]
    nrp = torch.zeros_like(row_ptr)
    torch.cumsum(nd, 0, out=nrp[1:])
    nsid = torch.empty_like(sid)
    ncon = torch.empty_like(conprb)
    CH = 5_000_000
    for a in range(0, N, CH):
        b = min(N, a + CH)
        ha, hb = int(nrp[a].item()), int(nrp[b].item())
        src = torch.repeat_interleave(row_ptr[perm[a:b]] - nrp[a:b], nd[a:b]) + torch.arange(ha, hb, device=sid.device)
        nsid[ha:hb] = sid[src]
        ncon[ha:hb] = conprb[src]
        del src
    return nrp, nsid, ncon, ncpv[perm].contiguous()


# --------------------------------------------------------------------------------------------------
def _ref_tools():
    exe = os.path.join(ROOT, "oracle", "_ref", "rsem-run-em-rounds")
    gen = os.path.join(ROOT, "tools", "gen_dataset")
    idx = os.path.join(ROOT, "oracle", "_ref", "rsem-build-read-index")
    return (exe, gen, idx) if all(os.path.exists(x) for x in (exe, gen, idx)) else None


def _gen_ref_dataset(d, gen, idx, rt, M, n_reads, deg, read_len):
    subprocess.check_call([gen, "--out", d, "--read-type", str(rt), "--M", str(M), "--N1", str(n_reads), "--N0",
                           str(n_reads // 20), "--avg-family", str(deg), "--read-len", str(read_len), "--seed", "11"],
                          stderr=subprocess.DEVNULL)
    files = ([f"{d}/s.temp/s_alignable_1.fq", f"{d}/s.temp/s_alignable_2.fq"] if rt == 3 else
             [f"{d}/s.temp/s_alignable.fq"] if rt == 1 else [f"{d}/s.temp/s_alignable.fa"])
    subprocess.check_call([idx, "32", str(rt & 1), "1", *files])
    with open(f"{d}/s.temp/s.dat") as f:
        return int(f.readline().split()[1])


def _time_ref_rounds(exe, d, rt, threads, first, steps):
    """reference rsem-run-em -p threads: wall-clock per frozen-conprb round from the time stamps of its own 'ROUND =' lines"""
    total = first + steps
    env = dict(os.environ, RSEM_MAX_ROUND=str(total), RSEM_MIN_ROUND=str(total))
    p = subprocess.Popen([exe, f"{d}/ref/r", str(rt), f"{d}/s", f"{d}/s.temp/s", f"{d}/s.stat/s", "-p", str(threads)],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, env=env, text=True, bufsize=1)
    stamps = {}
    for line in p.stdout:
        if line.startswith("ROUND = "):
            stamps[int(line.split(",")[0].split("=")[1])] = time.perf_counter()
    p.wait()
    return (stamps[first + steps] - stamps[first]) / steps, (stamps[10] - stamps[1]) / 9


def run_reference(args):
    """The reference's own CPU implementation (oracle/_ref/rsem-run-em-rounds = the unmodified EM.cpp with MAX/MIN_ROUND
    from the environment) on a bounded sample of the workload: same transcriptome, 1/10 of the reads (SURVEY.md 8(d)).
    The thread count is swept and the BEST one is reported; a second, 4x smaller sample separates the per-hit cost
    from the fixed per-round cost (thread create/join + the serial merge of nThreads count vectors, EM.cpp:373-389), so
    that the extrapolation to the full workload is explicit.  The frozen-conprb rounds never touch the reads, so the
    sample uses the shortest reads the model accepts (2 x 30 bases) to keep the model rounds 1-11 - which the unmodified
    binary has to run first - inside the time budget."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload if args.workload in WORKLOADS else "C3"
    N, M, deg, zipf = WORKLOADS[name]
    tools = _ref_tools()
    if tools is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref binaries or tools/gen_dataset missing"}))
        return
    exe, gen, idx = tools
    cores = os.cpu_count() or 1
    n_sample = min(N, args.ref_reads)
    n_small = max(1000, n_sample // 4)
    rt = 3 if name in ("C3", "C5") else (1 if name == "C2" else 0)
    rl = 30
    deg_eff = deg if deg else 27  # Zipf(1.1) <= 200 has mean 27
    threads = sorted({max(1, cores // 8), max(1, cores // 4), max(1, cores // 2), cores})
    first = 11 + args.warmup
    t_begin = time.perf_counter()
    with tempfile.TemporaryDirectory(prefix="rsem_ref_bench_") as d:
        H = _gen_ref_dataset(f"{d}/big", gen, idx, rt, M, n_sample, deg_eff, rl)
        sweep, model_s = {}, {}
        for p in threads:
            sweep[p], model_s[p] = _time_ref_rounds(exe, f"{d}/big", rt, p, first, args.steps)
            if time.perf_counter() - t_begin > args.ref_budget:  # keep the arm within its time budget
                break
        best = min(sweep, key=sweep.get)
        Hs = _gen_ref_dataset(f"{d}/small", gen, idx, rt, M, n_small, deg_eff, rl)
        small_s, _ = _time_ref_rounds(exe, f"{d}/small", rt, best, first, args.steps)
    s_per_round = sweep[best]
    per_hit = (s_per_round - small_s) / (H - Hs)
    fixed = s_per_round - per_hit * H
    full_hits = N * deg_eff
    value = H / s_per_round
    fit = {"ns_per_hit": round(per_hit * 1e9, 4), "fixed_ms_per_round": round(fixed * 1e3, 3),
           "samples": {str(H): round(s_per_round * 1e3, 3), str(Hs): round(small_s * 1e3, 3)},
           "extrapolated_full_workload_hits_per_s": full_hits / (fixed + per_hit * full_hits) if per_hit > 0 else None,
           "note": "t(round) = fixed + ns_per_hit * hits, from the two sample sizes at the best thread count"}
    sample = (f"{n_sample} of {N} reads / {H} hits (read_type {rt}, 2 x {rl} bases, all {M} transcripts) from tools/gen_dataset; "
              f"reference rsem-run-em -p {{{', '.join(str(p) for p in sweep)}}}: "
              + ", ".join(f"-p {p}: {H / sweep[p]:.3g} hits/s" for p in sweep)
              + f"; best -p {best}; rounds {first + 1}..{first + args.steps} timed from its ROUND lines; its model rounds 2-10 took "
              f"{model_s[best] * 1e3:.0f} ms each; whole arm {time.perf_counter() - t_begin:.0f} s")
    out = {"impl": "reference", "metric": "em_reads_hits_per_sec", "value": value, "unit": "hits/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_round * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": f"{name} (bounded sample: {n_sample} of {N} reads, all {M} transcripts)"},
           "cpu_baseline": {"value": value, "unit": "hits/s", "cores": best, "kind": "reference", "sample": sample,
                            "host_threads_available": cores, "thread_sweep_hits_per_s": {str(p): H / sweep[p] for p in sweep},
                            "fit": fit},
           "e2e": {"value": value, "unit": "hits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "head": git_head()}
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 20; MODEL times the model rounds 3-10 of rsem-run-em, so 8 there)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS) + ["C4", "MODEL"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: one shard of the workload per GPU (weak) or ONE matrix sharded over the GPUs (strong)")
    ap.add_argument("--scale", type=float, default=1.0, help="scale the number of reads (debugging only)")
    ap.add_argument("--variant", type=int, default=0, help="E-step kernel variant (0 auto, 4 row groups on CSR, 5 class layout)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sort-rows", default="", choices=["", "start", "deg"],
                    help="experiment: reorder the reads by first transcript id or by degree")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (kernel experiments)")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu child run that measures dram bytes per K2 launch")
    ap.add_argument("--traffic-probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--deg", type=int, default=0, help="experiment: override the mean number of hits per read")
    ap.add_argument("--ref-reads", type=int, default=5_000_000, help="reads in the reference arm's bounded sample")
    ap.add_argument("--ref-budget", type=float, default=240.0, help="seconds after which the reference arm stops sweeping threads")
    ap.add_argument("--gibbs-reads", type=int, default=10_000_000)
    ap.add_argument("--gibbs-chains", type=int, default=8)
    ap.add_argument("--model-reads", type=int, default=2_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned as DIR/<name>.npy: theta and the round statistics (EM "
                         "workloads), the last count vector of every chain and the posterior sums (C4)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload == "MODEL"):
        # MODEL times whole rsem-run-em processes: their outputs are files in a temporary directory, and the drop-in
        # tests compare those files with the reference's
        ap.error("--dump-outputs covers --impl ours with the EM workloads (C1, C2, C3, C5) and C4")
    if args.impl == "ours" and args.workload == "MODEL":
        # only rounds 1-10 of rsem-run-em update the model; rounds 1-2 carry the first launches, so 3-10 are timed
        if args.steps not in (None, 8):
            ap.error("--workload MODEL times the 8 model rounds 3-10 of rsem-run-em: --steps must be 8")
        args.steps = 8
    elif args.steps is None:
        args.steps = 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    # pin the OpenMP threads of the cpu_baseline leg before any OpenMP runtime starts
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "C4":
        import bench_extra
        bench_extra.run_gibbs(args)
    elif args.workload == "MODEL":
        import bench_extra
        bench_extra.run_model(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
