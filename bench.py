#!/usr/bin/env python
"""bench.py -- Step-1 level-0 ridge throughput (SNPs/s) on synthetic PLINK panels.

  python bench.py --gpus N --steps K --warmup W            # the B200 path (C ABI)
  python bench.py --impl reference --steps K --warmup W    # the CPU port of the reference path
  python bench.py --gpus 1 ... --dump-outputs DIR           # + what the last timed pass computed, DIR/*.npy

One "step" = one full level-0 pass (decode -> Gram -> ridge solves -> out-of-fold predictions
-> standardised W) over ALL blocks of the workload (BASELINE.json configs[1]: N=100k samples,
M=50k SNPs, 10 QTs, --bsize 1000, 5 folds, 5 ridge values, 3 covariates incl. intercept).
`value` is device-resident throughput; `e2e` feeds the same pass from pinned HOST .bed rows
through the C ABI (H2D inside the timed region) and reads the status word back.
With --gpus N (torchrun) the SAME pipeline runs sharded: one problem of N x 50 blocks on the same samples, SNP blocks
partitioned over the ranks by the reference's --split-l0 rule, every rank storing the predictor tiles of a phenotype
straight into the HBM of the rank that owns that phenotype's level 1 (CUDA IPC over NVLink, no collective on the data
path).  Per-GPU level-0 work is fixed (weak scaling in M); value = total SNPs / max time over ranks.  After the timed
level-0 passes the sharded level 1 (by phenotype) and the LOCO assembly run once and are reported beside it.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: nothing is written there
# Hardware queues for the lane streams of a Step-1 handle: with 32 instead of the driver's default 8 the library runs 12 lanes
# (csrc/rg_api.cu, rg_step1_create; profiles/ab_r2u_connections_lanes.txt).  The variable is read when the CUDA context is
# created, i.e. it has to be in the environment before torch touches the device.  A 32-queue context takes ~1 s longer to
# create, which a long job does not notice and a 1.3 s from-files run does: that leg's child process gets the default back.
_CONN_WAS_SET = "CUDA_DEVICE_MAX_CONNECTIONS" in os.environ
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

SEED = 20260924
CFG = dict(N=100_000, M=50_000, P=10, C=3, bsize=1000, K=5, R=5, miss=0.01)
DUMP_BYTES = 48 << 20                    # --dump-outputs: at most this much of W (a fixed, seeded sample of its rows)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ----------------------------------------------------------------------------- synthetic data
def gen_panel_gpu(torch, N, M, bsize, seed, device, miss):
    """Packed PLINK rows [M, ceil(N/4)] on the device: MAF~U(0.01,0.5), Binomial(2,MAF), `miss` NA."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    stride = (N + 3) // 4
    out = torch.empty((M, stride), dtype=torch.uint8, device=device)
    code = torch.tensor([3, 2, 0, 1], dtype=torch.uint8, device=device)   # dosage 0,1,2,NA -> PLINK code
    for s in range(0, M, bsize):
        bs = min(bsize, M - s)
        maf = torch.rand((bs, 1), generator=g, device=device) * 0.49 + 0.01
        d = (torch.rand((bs, N), generator=g, device=device) < maf).to(torch.uint8)
        d += (torch.rand((bs, N), generator=g, device=device) < maf).to(torch.uint8)
        if miss > 0:
            d[torch.rand((bs, N), generator=g, device=device) < miss] = 3
        c = code[d.long()]
        if N % 4:
            c = torch.nn.functional.pad(c, (0, 4 - N % 4))
        c = c.view(bs, stride, 4)
        out[s:s + bs] = c[:, :, 0] | (c[:, :, 1] << 2) | (c[:, :, 2] << 4) | (c[:, :, 3] << 6)
        del d, c
    return out


def gen_pheno(N, P, C, seed):
    rng = np.random.default_rng(seed)
    Y = rng.normal(size=(N, P))
    cov = rng.normal(size=(N, C - 1))
    na = rng.random(size=(N, P)) < 0.02
    return Y, cov, na


def blocks_of(M, bsize):
    return [(s, min(bsize, M - s)) for s in range(0, M, bsize)]


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip().split(", "))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        hi = [x for x in sm if mx and x > 0.3 * mx] or sm
        return {"sm_mhz": float(np.median(hi)) if hi else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU baseline (Eigen restatement)
def cpu_level0_blocks(packed_rows_list, N, X, Y, mask, in_an, fsz, lam, neff, threads=0):
    """Time the reference's level-0 path on the host cores: oracle/ref_eigen = C++ restatement of
    readChunkFromBedFileToG + residualize_genotypes + calc_cv_matrices + ridge_level_0 compiled against the
    reference's vendored Eigen 3.4.0 with -O3 -ffast-math -fopenmp (the reference binary itself cannot be built
    here: Boost / BGEN library absent).  Returns (SNPs, seconds, W of the first block, per-phase seconds)."""
    from oracle import ref_eigen             # the one place bench.py runs the oracle: the CPU baseline / parity check
    t0 = time.perf_counter()
    nsnp, W0, phases = 0, None, np.zeros(4)
    for rows in packed_rows_list:
        W, ph = ref_eigen.l0_block_kfold(rows, N, in_an, X, Y, mask, fsz, lam, neff, int(np.asarray(in_an).sum()),
                                         threads=threads)
        phases += ph
        if W0 is None:
            W0 = W
        nsnp += rows.shape[0]
    return nsnp, time.perf_counter() - t0, W0, phases


def calibrate_threads(rows, N, X, Y, mask, in_an, fsz, lam, neff):
    """Eigen's OpenMP GEMM does not scale to every hardware thread of a big host (128 threads: 94 s per block, slower
    than 8).  Time one block at a few thread counts and keep the fastest: the CPU arm gets its best configuration."""
    q = cpu_quota()
    if q:                                          # around the quota: fewer, exactly, and oversubscribed
        cands = sorted({max(1, q // 2), q, min(hw_threads(), 2 * q)})
    else:
        nthr = hw_threads()
        cands = sorted({max(1, nthr // 8), max(1, nthr // 4), max(1, nthr // 2)})
    if os.environ.get("OMP_NUM_THREADS"):          # torchrun pins this to 1; the CPU arm is a separate measurement
        os.environ.pop("OMP_NUM_THREADS")
    best, log = None, []
    for t in cands:
        _, dt, _, _ = cpu_level0_blocks([rows], N, X, Y, mask, in_an, fsz, lam, neff, threads=t)
        log.append("%d thr %.1f s" % (t, dt))
        if best is None or dt < best[1]:
            best = (t, dt)
    return best[0], "; ".join(log)


def cpu_baseline_desc(phases, dt, nblocks, bs, N, threads):
    from oracle import ref_eigen
    return ("%d block(s) of %d SNPs at N=%d from the same panel; C++ restatement of the reference's level-0 path on %s, "
            "%d OpenMP threads; %.1f s = decode+impute %.1f / residualise %.1f / cv matrices %.1f / eigensolver+ridge %.1f"
            % (nblocks, bs, N, ref_eigen.build_info(), threads, dt, phases[0], phases[1], phases[2], phases[3]))


def cpu_quota():
    """CPUs the container may use at once (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited.  The GPU boxes of this
    pool show 128 hardware threads but cpu.max = "1600000 100000": 16 CPUs - more threads than that only time-share."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return max(1, int(math.ceil(float(q) / float(per))))
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return max(1, int(math.ceil(q / per)))
    except Exception:
        pass
    return None


def hw_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def host_threads():
    """Threads the CPU arm can really run concurrently: hardware threads in the affinity mask, capped by the cgroup quota."""
    q = cpu_quota()
    return min(hw_threads(), q) if q else hw_threads()


def host_desc():
    q = cpu_quota()
    return "%d hardware threads visible, cgroup CPU quota %s" % (hw_threads(), ("%d CPUs" % q) if q else "none")


# ----------------------------------------------------------------------------- main arms
def run_reference(args):
    """--impl reference: the reference's CPU level-0 path (Eigen/OpenMP restatement, all host threads), one block per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from regenie_b200 import hostprep, synth
    c = CFG
    N, bs = c["N"], c["bsize"]
    Yr, cov, na = gen_pheno(N, c["P"], c["C"], SEED)
    X, Y, mask, in_an, neff = hostprep.prepare_qt(Yr, cov, na)
    fsz = hostprep.fold_sizes(N, c["K"])
    lam = c["M"] * (1 - hostprep.ridge_grid(c["R"])) / hostprep.ridge_grid(c["R"])
    n_steps = args.steps + args.warmup
    rows = [synth.pack_bed(synth.genotypes(N, bs, seed=SEED + i, miss=c["miss"])) for i in range(min(n_steps, 2))]
    times = []
    cores, calib = calibrate_threads(rows[0], N, X, Y, mask, in_an, fsz, lam, neff)
    phases = np.zeros(4)
    for i in range(n_steps):
        n, dt, _, ph = cpu_level0_blocks([rows[i % len(rows)]], N, X, Y, mask, in_an, fsz, lam, neff, threads=cores)
        if i >= args.warmup:
            times.append(dt)
            phases += ph
    tot = sum(times)
    val = bs * len(times) / tot
    line = {
        "impl": "reference", "metric": "step1_level0_snps_per_sec", "value": val, "unit": "SNPs/s",
        "n_gpus": 0, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": {"value": val, "unit": "SNPs/s", "cores": cores, "kind": "port",
                         "sample": "one 1000-SNP block per step; " + cpu_baseline_desc(phases, tot, len(times), bs, N, cores)
                                   + "; thread-count calibration on one block (fastest kept; %s): %s" % (host_desc(), calib)},
        "e2e": {"value": val, "unit": "SNPs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config():
    c = CFG
    return {"workload": "BASELINE.json configs[1]: synthetic PLINK .bed N=100k x M=50k, 10 QT, --step 1 --bsize 1000 "
                        "(level-0 ridge, 5 folds x 5 ridge values, 3 covariates, 1% missing calls)",
            "n_samples": c["N"], "n_snps": c["M"], "n_pheno": c["P"], "bsize": c["bsize"], "cv_folds": c["K"],
            "n_ridge_l0": c["R"], "l2_policy": "inputs larger than L2 (1.25 GB packed .bed per step, streamed once)",
            "parallelism": "snp-block sharding, no data-path collective"}


def run_gpu(args):
    import torch
    from regenie_b200 import capi, hostprep
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available() or capi.lib().rg_device_count() == 0:
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    c = CFG
    N, M, bs, P, C, K, R = c["N"], c["M"], c["bsize"], c["P"], c["C"], c["K"], c["R"]
    if args.small:
        N, M = 20_000, 4_000
    if args.n_samples:                      # exploration only (e.g. the N = 500k shape of configs[2] on a slice of blocks)
        N = args.n_samples
        M = (args.blocks or 20) * bs
    if args.n_pheno:                        # exploration only (the 50-trait shape of configs[4])
        P = args.n_pheno
    blocks = blocks_of(M, bs)
    if args.blocks:
        blocks = blocks[: args.blocks]
        M = sum(n for _, n in blocks)
    Yr, cov, na = gen_pheno(N, P, C, SEED)
    X, Y, mask, in_an, neff = hostprep.prepare_qt(Yr, cov, na)
    fsz = hostprep.fold_sizes(N, K)
    h = hostprep.ridge_grid(R)
    lam = M * (1 - h) / h
    panel = gen_panel_gpu(torch, N, M, bs, SEED + 1000 * rank, dev, c["miss"])
    stride = panel.shape[1]
    torch.cuda.synchronize()
    host_panel = torch.empty(panel.shape, dtype=torch.uint8, pin_memory=True)
    host_panel.copy_(panel)
    torch.cuda.synchronize()

    nb_local = len(blocks)
    st = capi.Step1(X, Y, mask, in_an, fsz, lam, neff, N, bs, nb_local * world, device=local)
    ext = torch.cuda.ExternalStream(st.stream(), device=dev)
    owner = None
    if world > 1:
        from regenie_b200 import sharding
        owner = sharding.attach_peers(st)       # W of phenotype p lives on rank p mod world; stores go over NVLink
    blk0 = rank * nb_local                      # this rank's contiguous block range of the global problem

    def one_pass(base_ptr):
        for b, (s, n) in enumerate(blocks):
            st.l0_block_bed(base_ptr + s * stride, n, blk0 + b, row_stride=stride)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(base_ptr, steps, read_status):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        barrier()
        l0 = st.launch_count()
        e0.record(ext)
        for _ in range(steps):
            one_pass(base_ptr)
            if read_status == "drain":
                bad = st.status() != 0        # waits for every block of the pass before the next pass is enqueued
            elif read_status:
                bad = st.poll_status() != 0   # 8-byte D2H read of the sticky error word beside the running lanes
            else:
                bad = False
            if bad:
                raise SystemExit("level-0 reported an error (timed/e2e pass): " + capi.lib().rg_last_error().decode())
        if read_status and st.status() != 0:  # the draining read: every block of every pass has reported by now
            raise SystemExit("level-0 reported an error (timed/e2e pass): " + capi.lib().rg_last_error().decode())
        st.fence()
        e1.record(ext)
        e1.synchronize()
        barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, st.launch_count() - l0

    dev_ptr, host_ptr = panel.data_ptr(), host_panel.data_ptr()
    for _ in range(max(args.warmup, 3)):
        one_pass(dev_ptr)
    if st.status() != 0:
        raise SystemExit("level-0 reported an error (warm-up): " + capi.lib().rg_last_error().decode())

    # ---- device-resident throughput (the timed region)
    clocks = ClockSampler(local); clocks.start()
    ms, launches = timed(dev_ptr, args.steps, read_status=False)
    clk = clocks.stop()
    st.sync()
    if st.status() != 0:
        raise SystemExit("level-0 reported an error (timed pass): " + capi.lib().rg_last_error().decode())
    if args.dump_outputs:
        dump_level0(st, len(blocks), N, P, R, args.dump_outputs)
    total_snps = M * args.steps * world
    value = total_snps / (ms / 1e3)

    # ---- per-kernel durations with CUDA events on the launching stream.  The timed region overlaps
    # consecutive blocks on several streams ("lanes"), so a kernel's event-bracketed time there includes
    # time-sharing with other kernels; for the roofline each kernel is ALSO timed alone (single lane).
    knames = ["bed_relayout", "bed_expand", "l0_stats", "gram_tcgen05", "l0_assemble", "mx_solve", "chol_factor",
              "chol_backsolve", "l0_predict"]

    def kernel_times(handle, nsteps):
        handle.set_timing(True)
        for _ in range(nsteps):
            for b, (s, n) in enumerate(blocks):
                handle.l0_block_bed(dev_ptr + s * stride, n, b, row_stride=stride)
        handle.sync()
        out = {}
        for k in knames:
            t, n = handle.timing(k)
            out[k] = {"ms_total": round(t, 3), "launches": n}
        handle.set_timing(False)
        return out

    kern_conc = kernel_times(st, 1)
    os.environ["RG_B200_LANES"] = "1"
    st1 = capi.Step1(X, Y, mask, in_an, fsz, lam, neff, N, bs, len(blocks), device=local)
    os.environ.pop("RG_B200_LANES", None)
    for b, (s, n) in enumerate(blocks[:4]):
        st1.l0_block_bed(dev_ptr + s * stride, n, b, row_stride=stride)
    st1.sync()
    kern = kernel_times(st1, 1)
    st1.close()

    # ---- end to end: pinned host rows -> H2D -> same pass -> status word D2H, every step
    for _ in range(1):
        one_pass(host_ptr)
    ms_e2e, _ = timed(host_ptr, args.steps, read_status=os.environ.get("RG_BENCH_E2E_STATUS", "poll"))   # env "drain": A/B only
    e2e_val = total_snps / (ms_e2e / 1e3)

    # ---- the rest of the sharded Step 1, once: level 1 by phenotype on the owners, LOCO assembly, gather to all ranks
    sharded = None
    if world > 1:
        from regenie_b200 import sharding
        st.sync(); barrier()
        Bt = nb_local * world * R
        h1 = hostprep.ridge_grid(5)
        tau = np.tile(Bt * (1 - h1) / h1, (P, 1))
        chr_of_block = [1 + (22 * b) // (nb_local * world) for b in range(nb_local * world)]
        # the level-1 / LOCO work of this rank; a failure here (a width B = nb x world x R this build has not met on hardware)
        # must not take the level-0 numbers of the run with it: every rank learns whether any rank failed before the gathers
        l1_err, t_l1, t_loco = None, 0.0, 0.0
        try:
            t0 = time.perf_counter()
            cs, best = st.l1_fit(tau)
            t_l1 = time.perf_counter() - t0
            t0 = time.perf_counter()
            loco = st.loco(chr_of_block)
            t_loco = time.perf_counter() - t0
        except Exception as e:
            l1_err = "rank %d: %s" % (rank, str(e)[:200])
        flag = torch.tensor([1.0 if l1_err else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if float(flag.item()) > 0:
            sharded = {"error": l1_err or "level 1 / LOCO failed on another rank", "level1_width_B": Bt}
        else:
            t0 = time.perf_counter()
            cs = sharding._sum_to_all(cs, dev); loco = sharding._sum_to_all(loco, dev)
            t_gather = time.perf_counter() - t0
            tt = torch.tensor([t_l1, t_loco, t_gather], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            n_owned = sum(1 for p in range(P) if owner[p] == rank)
            peer_bytes = nb_local * R * N * 8 * (P - n_owned)                          # W columns stored to other ranks per pass
            pb = torch.tensor([float(peer_bytes)], dtype=torch.float64, device=dev)
            dist.all_reduce(pb, op=dist.ReduceOp.MAX)
            sharded = {"level1_seconds": float(tt[0]), "loco_seconds": float(tt[1]), "gather_seconds": float(tt[2]),
                       "level1_width_B": Bt, "phenotypes_per_rank_max": max(owner.count(r) for r in range(world)),
                       "peer_store_bytes_per_rank_per_step": float(pb[0]),
                       "peer_store_GBps_per_rank": float(pb[0]) / (ms / args.steps * 1e-3) / 1e9,
                       "nvlink_peer_copy_reference_GBps": 770.0,
                       "finite": bool(np.isfinite(cs).all() and np.isfinite(loco).all()),
                       "note": "level 1 is sharded by phenotype (p mod world): with %d traits on %d ranks the busiest rank fits %d; "
                               "stores to peers ride inside the prediction / standardisation kernels, overlapped with compute"
                               % (P, world, max(owner.count(r) for r in range(world)))}

    # ---- end to end from files through the C++ driver (rank 0, single GPU run only)
    file_e2e = None
    if world == 1 and not args.no_step2 and not (args.small or args.n_samples or args.blocks or args.n_pheno):
        try:
            file_e2e = file_e2e_leg(host_panel, N, M, bs, P, Yr, cov, na)
        except Exception as e:
            file_e2e = {"error": str(e)[:300]}

    # ---- second half of the metric: Step-2 variants/s (QT on .bed rows, BT on 8-bit BGEN dosages), each with a
    # host-fed rate, a device-resident rate, an HBM roofline and a CPU baseline (rank 0 only)
    s2 = None
    if not args.no_step2 and rank == 0:
        try:
            s2 = step2_qt_leg(capi, X, mask, in_an, N, P, C, bs, blocks, host_panel, dev_ptr, stride, args)
        except Exception as e:          # never let the secondary metric break the headline line
            s2 = {"error": str(e)[:300]}
        try:
            s2["bt_bgen"] = step2_bt_leg(capi, X, in_an, N, C, args)
        except Exception as e:
            s2["bt_bgen"] = {"error": str(e)[:300]}
        try:
            s2["pgen_decode"] = pgen_decode_leg(capi, X, in_an, N, args)
        except Exception as e:
            s2["pgen_decode"] = {"error": str(e)[:300]}

    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return
    peaks, peak_src = load_peaks()
    gram_ms, gram_n = kern["gram_tcgen05"]["ms_total"], max(1, kern["gram_tcgen05"]["launches"])
    flops_per_launch = 2.0 * bs * bs * N          # SURVEY 8(d): 2*N*bs per SNP x bs SNPs (reference src/Data.cpp:748)
    ach = flops_per_launch / (gram_ms / gram_n * 1e-3) / 1e12
    # the Gram runs in e4m3 (exact for hard calls); FP8 dense peak = 2 x the measured BF16 cuBLAS rate
    peak_bf16 = peaks.get("bf16_tflops") or peaks.get("bf16_tflops_sustained")   # kernel timed alone -> burst figure
    peak = 2.0 * peak_bf16
    ktot = sum(v["ms_total"] for v in kern.values()) or 1.0
    for v in kern.values():
        v["share"] = round(v["ms_total"] / ktot, 4)
    # FP64 solver: K*R Cholesky factorisations of bs x bs per block
    solver_ms_tot = kern["mx_solve"]["ms_total"] + kern["chol_factor"]["ms_total"] + kern["chol_backsolve"]["ms_total"]
    solver_n = max(1, kern["mx_solve"]["launches"], kern["chol_factor"]["launches"])
    chol_ms = solver_ms_tot / solver_n
    chol_tf = (K * R * bs ** 3 / 3.0) / (chol_ms * 1e-3) / 1e12 if chol_ms > 0 else None
    mixed_blocks, f64_fallbacks = st.solver_stats()

    # step-level roofline (SURVEY 8d): algorithmic flops per SNP F0 = 2 N bs + 2 N P (1 + R) + 4 N C, whole-job rate
    F0 = 2.0 * N * bs + 2.0 * N * P * (1 + R) + 4.0 * N * C
    step_tf = value * F0 / 1e12 / world
    peak_sust = 2.0 * (peaks.get("bf16_tflops_sustained") or peak_bf16)
    traffic, pipe_active = gram_traffic_from_profile()
    cpu, parity = None, None
    if not args.no_cpu:
        rows = [host_panel[s:s + n].numpy() for (s, n) in blocks[: args.cpu_blocks]]
        thr, calib = calibrate_threads(rows[0], N, X, Y, mask, in_an, fsz, lam, neff)
        nsnp, dt, W_cpu, phases = cpu_level0_blocks(rows, N, X, Y, mask, in_an, fsz, lam, neff, threads=thr)
        cpu = {"value": nsnp / dt, "unit": "SNPs/s", "cores": thr, "kind": "port",
               "sample": cpu_baseline_desc(phases, dt, len(rows), bs, N, thr)
                         + "; thread-count calibration on one block (fastest kept; %s): %s" % (host_desc(), calib)}
        # parity on the benchmarked configuration: block 0 of the timed panel, every predictor column, GPU vs Eigen
        err = 0.0
        for p in range(P):
            Wg = st.fetch_W(0, p)
            err = max(err, float(np.abs(Wg - W_cpu[p]).max() / np.abs(W_cpu[p]).max()))
        parity = {"max_rel_err": err, "tol": 1e-9, "what": "level-0 predictors W of block 0 (N x %d columns x %d traits) of the "
                  "timed panel, B200 path vs the Eigen restatement of ridge_level_0" % (R, P)}
        if not (err < 1e-9):
            raise SystemExit("bench.py: parity check failed on the benchmarked configuration: max rel err %g" % err)

    line = {
        "metric": "step1_level0_snps_per_sec", "value": value, "unit": "SNPs/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "e4m3 Gram + int8 prediction (both exact integer sums) + tf32x3 factorisation + f64 refinement / statistics",
        "data": "synthetic", "config": workload_config() if not (args.small or args.n_samples or args.n_pheno) else {"workload": "NOT the benchmark configuration (smoke / exploration run)", "n_samples": N, "n_snps": M, "n_pheno": P},
        "clocks": clk,
        "e2e": {"value": e2e_val, "unit": "SNPs/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(M) * int(stride), "d2h_bytes_per_step": 8,
                "result_read": "every pass: rg_l0_poll_status (8-byte D2H read of the sticky error word, lanes keep running); "
                               "after the last pass, inside the timed region: rg_l0_status (waits for every block)"},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "gram_fp8_tcgen05_kernel", "bound": "tensor", "achieved": ach, "peak": peak,
                     "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic,
                     "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full "
                                     "(profiles/ncu_r2o_key_kernels.txt, else ncu_r1n_key_kernels.txt); algorithmic bytes = 205 MB of "
                                     "Z planes + 47 MB of Gram tiles",
                     "executed_frac": 2.0 * ach / peak, "tensor_pipe_active_ncu": pipe_active,
                     "peak_basis": "2 x %s bf16 cuBLAS rate (%s TF/s) = dense FP8" % (peak_src, peak_bf16),
                     "algorithmic_flops_per_launch": flops_per_launch,
                     "timed": "alone (single lane), CUDA events on the launching stream",
                     "note": "kernel executes 2x this (lower triangle of the [G0;Miss] Gram) to handle missing calls exactly"},
        "step_roofline": {"flops_per_snp": F0, "achieved_tflops_per_gpu": step_tf, "peak": peak_sust, "frac": step_tf / peak_sust,
                          "peak_basis": "2 x %s SUSTAINED bf16 cuBLAS rate = dense FP8, kernel mix timed inside a long step" % peak_src,
                          "note": "whole level-0 step (decode, statistics, Gram, solver, predictions) against the tensor "
                                  "roofline of its algorithmic flops; the solver's share is in `solver`"},
        "solver": {"kernel": "mixed: 3xTF32 tcgen05 factorisation / inverse + FP64 refinement (chol_mixed.cu)" if mixed_blocks else
                             "fp64: DMMA Cholesky + back-substitution (chol.cu)",
                   "ms_per_block_single_lane": chol_ms,
                   "cholesky_equivalent_tflops": chol_tf,
                   "note": "K*R*bs^3/3 flops of one Cholesky per system divided by the solver's time (the mixed path executes ~3x "
                           "that in TF32 products plus the FP64 refinement passes); FP64 pipe nominal 40 TF/s for scale",
                   "blocks_mixed": mixed_blocks, "blocks_fp64_fallback": f64_fallbacks,
                   "share_of_single_lane_kernel_time": round(solver_ms_tot / ktot, 4)},
        "kernels": kern,
        "kernels_concurrent": kern_conc,
        "lanes": int(os.environ.get("RG_B200_LANES", "12" if int(os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS", "8")) >= 16 else "8")),
        "cuda_device_max_connections": int(os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS", "8")),
        "cpu_baseline": cpu,
        "sharded_step1": sharded,
        "from_files": file_e2e,
        "parity": parity,
        "step2": s2,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


def dump_level0(st, nblocks, N, P, R, d):
    """What the last timed pass computed, as a caller of rg_l0_fetch_W receives it: the level-0 predictors W (N x R per
    block and phenotype).  All of W is nblocks x P x N x R doubles (2 GB for the benchmark), so the same seeded sample of
    rows is kept from every block: level0_W.npy [nblocks, P, rows, R] float64, the row indices in level0_W_rows.npy."""
    n_rows = max(1, min(N, DUMP_BYTES // (8 * nblocks * P * R)))
    rows = np.sort(np.random.default_rng(SEED).choice(N, n_rows, replace=False))
    W = np.empty((nblocks, P, n_rows, R))
    for b in range(nblocks):
        for p in range(P):
            W[b, p] = st.fetch_W(b, p)[rows]
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "level0_W.npy"), W)
    np.save(os.path.join(d, "level0_W_rows.npy"), rows.astype(np.float64))


def file_e2e_leg(host_panel, N, M, bs, P, Yr, cov, na, gpus=1):
    """End to end FROM FILES through the C++ driver: write the benchmark panel as a real PLINK fileset + phenotype /
    covariate text files, run `rgb200 --step 1` (reader thread -> rg_l0_block_bed -> level 1 -> LOCO -> .loco text) and
    time the whole process.  This is the reference's own user-facing path (regenie --step 1 --bed ... --out ...)."""
    import tempfile
    rgb = os.path.join(ROOT, "regenie_b200", "rgb200")
    d = tempfile.mkdtemp(prefix="rgbench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        t0 = time.perf_counter()
        with open(os.path.join(d, "p.bed"), "wb") as fh:
            fh.write(b"\x6c\x1b\x01")
            fh.write(host_panel.numpy().tobytes())
        per = (M + 21) // 22
        with open(os.path.join(d, "p.bim"), "w") as fh:
            fh.write("".join("%d rs%d 0 %d A G\n" % (i // per + 1, i, 1000 + i) for i in range(M)))
        with open(os.path.join(d, "p.fam"), "w") as fh:
            fh.write("".join("F%d I%d 0 0 %d -9\n" % (s, s, 1 + s % 2) for s in range(N)))
        Yt = np.where(na, np.nan, Yr)
        with open(os.path.join(d, "pheno.txt"), "w") as fh:
            fh.write("FID IID " + " ".join("Y%d" % (p + 1) for p in range(P)) + "\n")
            for s_ in range(N):
                fh.write("F%d I%d " % (s_, s_) + " ".join("NA" if na[s_, p] else "%.17g" % Yt[s_, p] for p in range(P)) + "\n")
        with open(os.path.join(d, "covar.txt"), "w") as fh:
            fh.write("FID IID " + " ".join("V%d" % (c + 1) for c in range(cov.shape[1])) + "\n")
            for s_ in range(N):
                fh.write("F%d I%d " % (s_, s_) + " ".join("%.17g" % v for v in cov[s_]) + "\n")
        t_write = time.perf_counter() - t0
        cmd = [rgb, "--step", "1", "--bed", os.path.join(d, "p"), "--phenoFile", os.path.join(d, "pheno.txt"), "--covarFile",
               os.path.join(d, "covar.txt"), "--bsize", str(bs), "--out", os.path.join(d, "fit")]
        if gpus > 1:
            cmd += ["--gpus", str(gpus)]
        t0 = time.perf_counter()
        child_env = dict(os.environ, RG_B200_PHASES="1")
        if not _CONN_WAS_SET:
            child_env.pop("CUDA_DEVICE_MAX_CONNECTIONS", None)      # short job: default queue count (fast context creation), 8 lanes
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=child_env)
        dt = time.perf_counter() - t0
        if r.returncode != 0:
            return {"error": (r.stdout + r.stderr)[-300:]}
        phases = {}                                        # the driver's own wall clock per phase (stderr, RG_B200_PHASES)
        for l in r.stderr.splitlines():
            if l.startswith("[phase]") and "(+" in l:
                phases[l[7:].split("  ")[0].strip()] = float(l.split("(+")[1].split(")")[0])
        l0 = [l for l in r.stdout.splitlines() if "Level 0 done" in l]
        l0_ms = float(l0[0].split("(")[1].split("ms")[0]) if l0 else None
        ok = all(os.path.exists(os.path.join(d, "fit_%d.loco" % (p + 1))) for p in range(P))
        return {"metric": "step1_from_files_snps_per_sec", "value": M / dt, "unit": "SNPs/s", "seconds": dt,
                "level0_seconds_driver_log": None if l0_ms is None else l0_ms / 1e3,
                "level0_snps_per_sec_driver_log": None if not l0_ms else M / (l0_ms / 1e3),
                "loco_files_written": ok, "fileset_write_seconds": t_write, "phase_ms": phases,
                "what": "rgb200 --step 1 --bed (1.25 GB .bed in /dev/shm) --phenoFile --covarFile --bsize %d --out: process start to exit, "
                        "i.e. text parsing, phenotype preparation, level 0 from the file, level 1 (B = %d), LOCO and the %d .loco files"
                        % (bs, (M // bs) * 5, P)}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def step2_traffic_from_profile(kernels, variants_per_launch):
    """DRAM bytes per variant (dram__bytes_read.sum + dram__bytes_write.sum of one launch of each named kernel, divided by the
    variants a launch covers) from the committed ncu --set full summary of the Step-2 kernels (tools/ncu_capture_s2.sh ->
    profiles/ncu_r2t_step2_kernels.txt; captured at N = 100k: 1000 .bed variants / 400 dosage variants per launch)."""
    try:
        blocks = open(os.path.join(ROOT, "profiles", "ncu_r2t_step2_kernels.txt")).read().split("---\n")
    except OSError:
        return None, None
    per = {}
    for b in blocks:                                   # the LAST captured launch of each kernel (warm handle)
        name = next((k for k in kernels if k in b), None)
        if name is None:
            continue
        d = {}
        for line in b.splitlines():
            t = line.split()
            if len(t) >= 2:
                d[t[0]] = t[1]
        if "dram__bytes_read.sum" in d:
            per[name] = (float(d["dram__bytes_read.sum"]) + float(d["dram__bytes_write.sum"])) * 1e6 / variants_per_launch
    if len(per) != len(kernels):
        return None, None
    return sum(per.values()), {k: round(v) for k, v in per.items()}


def hbm_roofline(rate, bytes_per_variant, what, traffic=(None, None)):
    peaks, src = load_peaks()
    gbs = rate * bytes_per_variant / 1e9
    out = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
           "traffic": traffic[0], "algorithmic_bytes_per_variant": bytes_per_variant, "peak_basis": "%s copy bandwidth" % src,
           "rate_used": "device-resident variants/s x algorithmic bytes per variant (%s)" % what}
    if traffic[0] is not None:
        out["traffic_unit"] = "DRAM bytes per variant, all kernels of a block (ncu --set full at N = 100k, profiles/ncu_r2t_step2_kernels.txt)"
        out["traffic_by_kernel"] = traffic[1]
    return out


def s2_tensor_roofline(rate, N, P, C):
    """What really bounds the hard-call Step-2 path: with per-trait masks a variant needs D = 1 + C + 2P + PC exact sums over
    its N calls (not one pass over N/4 bytes), done as FP8 tensor tiles against 9 radix-30 digit rows per feature column for the
    three planes g0, g0^2, missing (csrc/s2_kernels.cu, s2_api.cu: digit rows padded to 14 columns per 128-row group)."""
    peaks, src = load_peaks()
    D = 1 + C + 2 * P + P * C
    drows = int(math.ceil(math.ceil(D / 14.0) * 128 / 256.0) * 256)
    executed = 2.0 * N * 3 * drows                      # flops per variant on the tensor pipe
    peak = 2.0 * (peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops"))
    tf = rate * executed / 1e12
    return {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
            "executed_flops_per_variant": executed, "feature_columns": D, "digit_rows": drows,
            "algorithmic_flops_per_variant": 2.0 * N * D,
            "peak_basis": "2 x %s sustained bf16 cuBLAS rate = dense FP8" % src,
            "note": "the HBM line above is SURVEY 8(d)'s scan bound (N/4 bytes per variant); at %d traits the exact digit-plane "
                    "tiles are the binding resource, not the bytes" % P}


def step2_qt_leg(capi, X, mask, in_an, N, P, C, bs, blocks, host_panel, dev_ptr, stride, args):
    """Step-2 QT score test on the benchmark panel's .bed rows (compute_score_qt, src/Step2_Models.cpp:343-467)."""
    from oracle import ref_eigen
    rng = np.random.default_rng(SEED + 7)
    res = np.asfortranarray(rng.normal(size=(N, P)) * mask)
    res /= np.linalg.norm(res, axis=0) / np.sqrt(mask.sum(axis=0) - C)
    st2 = capi.Step2(X, mask, in_an, N, bs)
    st2.set_chr(res, np.ones(P))
    nb2 = min(len(blocks), 10)
    out = st2._out(bs)
    hbase = host_panel.data_ptr()
    for b in range(2):                                              # warm-up (allocations, tensor maps)
        st2.block_bed_raw(hbase + blocks[b][0] * stride, blocks[b][1], stride, out)
        st2.block_bed_raw(dev_ptr + blocks[b][0] * stride, blocks[b][1], stride, out)

    def run(base):
        t0 = time.perf_counter(); nv = 0
        for b in range(nb2):
            st2.block_bed_raw(base + blocks[b][0] * stride, blocks[b][1], stride, out)
            nv += blocks[b][1]
        return nv / (time.perf_counter() - t0)
    host_rate = run(hbase)
    dev_rate = run(dev_ptr)

    def run_staged():
        # the rows of block b+1 cross PCIe (rg_s2_stage, copy stream) while block b is tested
        t0 = time.perf_counter(); nv = 0
        nxt = st2.stage(0, hbase + blocks[0][0] * stride, blocks[0][1] * stride)
        for b in range(nb2):
            cur = nxt
            if b + 1 < nb2:
                nxt = st2.stage((b + 1) & 1, hbase + blocks[b + 1][0] * stride, blocks[b + 1][1] * stride)
            st2.block_bed_raw(cur, blocks[b][1], stride, out)
            nv += blocks[b][1]
        return nv / (time.perf_counter() - t0)
    run_staged()
    staged_rate = run_staged()
    st2.close()
    # CPU: the Eigen restatement, one OpenMP task per variant like Data::test_snps_fast
    cpu = None
    if not args.no_cpu:
        nv_cpu = 8192                                  # ~ a few seconds of CPU work on the host cores
        rows = host_panel[:nv_cpu].numpy()
        YtX = res.T @ X
        thr = host_threads()
        ref_eigen.s2_block_qt_bed(rows[:32], N, in_an, X, res, mask, YtX, np.ones(P), int(in_an.sum()), threads=thr)
        t0 = time.perf_counter()
        ref_eigen.s2_block_qt_bed(rows, N, in_an, X, res, mask, YtX, np.ones(P), int(in_an.sum()), threads=thr)
        dt = time.perf_counter() - t0
        cpu = {"value": nv_cpu / dt, "unit": "variants/s", "cores": thr, "kind": "port",
               "sample": "%d variants at N=%d, %d traits: C++/Eigen restatement of parseSnpfromBed + residualize_geno + "
                         "compute_score_qt, one OpenMP task per variant (%.2f s)" % (nv_cpu, N, P, dt)}
    return {"metric": "step2_qt_variants_per_sec", "value": dev_rate, "unit": "variants/s",
            "e2e": {"value": max(host_rate, staged_rate), "unit": "variants/s", "h2d_bytes_per_variant": int(stride),
                    "d2h_bytes_per_variant": 8 * (6 * P + 3) + 4 * (P + 2),
                    "staged": staged_rate, "unstaged": host_rate,
                    "note": "staged = rg_s2_stage copies block b+1 on a copy stream under the kernels of block b; unstaged = "
                            "the block call copies its own rows first"},
            "roofline": hbm_roofline(dev_rate, N / 4.0, "N/4 bytes of 2-bit calls",
                                     step2_traffic_from_profile(("bed_relayout_kernel", "bed_expand3_fp8_kernel", "gram_fp8_tcgen05_kernel",
                                                                 "s2_stats_finish_kernel", "s2_finalize_kernel"), 1000) if N == 100_000 else (None, None)),
            "tensor_roofline": s2_tensor_roofline(dev_rate, N, P, C),
            "cpu_baseline": cpu,
            "sample": "%d blocks of %d variants, N=%d, %d traits; value = .bed rows resident in HBM, e2e = pinned host rows; "
                      "both through rg_s2_block_bed (synchronous call, per-variant statistics copied back every block)" % (nb2, bs, N, P)}


def pgen_decode_leg(capi, X, in_an, N, args, nvar=512):
    """SURVEY 8 (f)3: a block of .pgen records (host bytes) -> PLINK 1 rows in HBM through rg_pgen_decode, timed on the host
    around the synchronous Step-2 entry point (H2D of the record bytes + both kernels + status word), against the
    reference's own reader - the vendored pgenlib compiled from the reference sources (oracle/_ref/libpgenlib_ref.so),
    ReadHardcalls per variant as src/Geno.cpp:1798 calls it.  Parity: the rows fetched back equal the calls written."""
    import tempfile
    from regenie_b200 import synth
    rng = np.random.default_rng(17)
    g = np.zeros((nvar, N), dtype=np.uint8)
    for v in range(nvar):                                     # allele-frequency spectrum of an array / WES panel: mostly rare
        u = rng.random()
        maf = 10 ** rng.uniform(-4, -2) if u < 0.6 else (rng.uniform(0.01, 0.05) if u < 0.85 else rng.uniform(0.05, 0.5))
        if v and rng.random() < 0.15:                         # in LD with its neighbour: an LD-compressed record
            g[v] = g[v - 1]
            idx = rng.integers(0, N, 40)
            g[v][idx] = rng.binomial(2, 0.3, idx.size)
            continue
        g[v] = rng.binomial(2, maf, N)
        g[v][rng.random(N) < 0.002] = 3
    d = tempfile.mkdtemp(prefix="rgpgen_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        recs = []
        types = synth.write_pgen(os.path.join(d, "p"), g, storage=6, records_out=recs)
        b = synth.gather_pgen_records(lambda v: recs[v], lambda v: types[v], list(range(nvar)))
        st = capi.Step2(X, np.ones((N, 1), dtype=np.uint8), in_an, int(in_an.sum()), nvar, strict=True)
        for _ in range(3):
            rows, stride = capi.pgen_decode(st, n_file=N, **b)
        reps = 20
        t0 = time.perf_counter()
        for _ in range(reps):
            capi.pgen_decode(st, n_file=N, **b)
        dt = (time.perf_counter() - t0) / reps
        got = capi.debug_fetch(st, "pgen_rows", np.uint8, nvar * stride).reshape(nvar, stride)
        codes = np.stack([(got >> (2 * k)) & 3 for k in range(4)], axis=-1).reshape(nvar, -1)[:, :N]
        exact = bool(np.array_equal(codes, np.array([3, 2, 0, 1], dtype=np.uint8)[g]))
        st.close()
        if not exact:
            raise SystemExit("bench.py: device-decoded .pgen rows differ from the calls that were written")
        in_bytes, out_bytes = int(b["data"].size), nvar * ((N + 3) // 4)
        peaks, src = load_peaks()
        gbs = (in_bytes + out_bytes) / dt / 1e9
        cpu = None
        if not args.no_cpu:
            from oracle import pgenlib_ref
            if pgenlib_ref.available():
                ref, sec = pgenlib_ref.read_hardcalls(os.path.join(d, "p.pgen"), N, 0, nvar, timing=True)
                want = g.astype(float); want[want == 3] = -3.0
                if not np.array_equal(ref, want):
                    raise SystemExit("bench.py: pgenlib and the synthetic .pgen disagree")
                cpu = {"value": nvar / sec, "unit": "variants/s", "cores": 1, "kind": "reference",
                       "sample": "%d variants at N=%d through the reference's vendored pgenlib (PgenReader::ReadHardcalls per "
                                 "variant, one thread; the reference runs this loop under OpenMP), %.3f s" % (nvar, N, sec)}
        return {"metric": "pgen_decode_variants_per_sec", "value": nvar / dt, "unit": "variants/s", "ms_per_block": dt * 1e3,
                "record_bytes_per_variant": in_bytes / nvar, "row_bytes_per_variant": out_bytes / nvar,
                "record_types": {str(t): int(types.count(t)) for t in sorted(set(types))},
                "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                             "traffic": None, "peak_basis": src,
                             "note": "record bytes in + 2-bit rows out per block over the host-timed call (PCIe copy of the "
                                     "records, two kernels, status word): latency-bound at this block size, not HBM-bound"},
                "parity": {"bit_exact": exact, "what": "all %d rows fetched back from HBM vs the calls written" % nvar},
                "cpu_baseline": cpu,
                "sample": "%d variants at N=%d, 60 %% with MAF < 1 %%, 0.2 %% missing calls; host record bytes -> rows resident in HBM" % (nvar, N)}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def bgen_payloads(N, nvar, seed):
    """Imputed-looking 8-bit probability pairs + their BGEN v1.2 layout-2 payloads, zlib level 6 like qctool writes."""
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    rng = np.random.default_rng(seed)
    probs = np.zeros((nvar, N, 2), dtype=np.uint8)
    for v, maf in enumerate(rng.uniform(0.01, 0.5, nvar)):
        g = rng.binomial(2, maf, N)
        probs[v, g == 2, 0] = 255
        probs[v, g == 1, 1] = 255
        u = rng.random(N) < 0.15                                   # 15 % of calls are uncertain
        a = rng.integers(0, 256, int(u.sum()))
        probs[v, u, 0] = a
        probs[v, u, 1] = (rng.random(int(u.sum())) * (255 - a)).astype(np.uint8)
    hdr = np.zeros(8, dtype=np.uint8)
    hdr[:4] = np.frombuffer(np.uint32(N).tobytes(), dtype=np.uint8)
    hdr[4], hdr[6], hdr[7] = 2, 2, 2
    pl = np.full(N, 2, dtype=np.uint8)
    tail = np.array([0, 8], dtype=np.uint8)
    raws = [np.concatenate([hdr, pl, tail, probs[v].reshape(-1)]).tobytes() for v in range(nvar)]
    with ThreadPoolExecutor(16) as ex:
        comps = list(ex.map(lambda r: zlib.compress(r, 6), raws))
    offs = np.zeros(nvar + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(c) for c in comps])
    return probs, np.frombuffer(b"".join(comps), dtype=np.uint8), offs


def step2_bt_leg(capi, X, in_an, N, C, args, nvar=400, nblocks=4):
    """Step-2 binary-trait score test + approximate Firth on 8-bit BGEN dosages (BASELINE configs[3] shape at this N,
    compute_score_bt src/Step2_Models.cpp:470-556): pinned host probability bytes, bytes resident in HBM, and
    compressed payloads inflated on the device (both inflate kernels) in front of the same score test."""
    import torch
    from oracle import ref_eigen
    rng = np.random.default_rng(SEED + 11)
    y = (rng.random(N) < 0.1).astype(np.float64)                       # prevalence 10 %
    mask = np.ones((N, 1), dtype=np.uint8)
    p0 = float(y.mean())
    eta = math.log(p0 / (1 - p0))
    w = math.sqrt(p0 * (1 - p0))
    gsm = np.full((N, 1), w); yres = ((y - p0) / w)[:, None]
    # X is orthonormal with the intercept in its span: X_Gamma = X for a constant weight
    st = capi.Step2(X, mask, in_an, N, nvar)
    st.set_chr_bt(gsm, gsm, yres, [X], y[:, None], np.full((N, 1), eta))
    probs_np, comp, offs = bgen_payloads(N, nvar, SEED + 13)
    probs_t = torch.from_numpy(probs_np).pin_memory()
    miss_t = torch.full((nvar, N), 0x02, dtype=torch.uint8).pin_memory()
    probs_d, miss_d = probs_t.cuda(), miss_t.cuda()
    out = st._out(nvar, with_info=True)

    def block(pp, mp):
        o = st.block_bgen8_bt_raw(pp, mp, N, nvar, out)
        sel = np.nonzero((np.abs(o["stat"][:, 0]) > 1.959964) & ((o["flags"] & 17) == 0))[0]
        st.firth(sel, np.zeros(len(sel), dtype=np.int32))
        return len(sel)

    block(probs_t.data_ptr(), miss_t.data_ptr())                       # warm-up: scratch allocation

    def run(fn):
        t0 = time.perf_counter(); nf = 0
        for _ in range(nblocks):
            nf += fn()
        return nblocks * nvar / (time.perf_counter() - t0), nf / (nblocks * nvar)
    host_rate, ff = run(lambda: block(probs_t.data_ptr(), miss_t.data_ptr()))
    dev_rate, _ = run(lambda: block(probs_d.data_ptr(), miss_d.data_ptr()))
    # staged: the (same) pinned bytes of the NEXT block cross PCIe on the copy stream while this block is tested
    stage_state = {"n": 0, "next": None}

    def staged_block():
        k = stage_state["n"]
        if stage_state["next"] is None:
            stage_state["next"] = (st.stage(0, probs_t.data_ptr(), probs_t.numel()), st.stage(1, miss_t.data_ptr(), miss_t.numel()))
        cur = stage_state["next"]
        sl = 2 * ((k + 1) & 1)
        stage_state["next"] = (st.stage(sl, probs_t.data_ptr(), probs_t.numel()), st.stage(sl + 1, miss_t.data_ptr(), miss_t.numel()))
        stage_state["n"] = k + 1
        return block(cur[0], cur[1])
    staged_block()
    staged_rate, _ = run(staged_block)
    inflate = {}
    for mode in ("direct", "window"):
        os.environ["RG_B200_INFLATE"] = mode
        try:
            def fn():
                pd, md = st.bgen_inflate(comp, offs, N)
                return block(pd, md)
            fn()
            r, _ = run(fn)
            t0 = time.perf_counter()
            for _ in range(nblocks):
                st.bgen_inflate(comp, offs, N)
            ti = (time.perf_counter() - t0) / nblocks
            inflate[mode] = {"variants_per_sec_with_score_test": r, "inflate_ms_per_block": 1e3 * ti,
                             "inflated_GBps": nvar * (10 + 3 * N) / ti / 1e9}
        except Exception as e:
            inflate[mode] = {"error": str(e)[:200]}
    os.environ.pop("RG_B200_INFLATE", None)
    st.close()
    # one warp owns one stream and a stream takes ~27 ms whatever else runs: the inflate kernel's throughput is the number
    # of streams in flight.  Same payloads, one launch over 4096 of them (the 400 streams repeated) through a handle with
    # that block size - what `rgb200 --gpu-inflate --bsize 4096` does
    try:
        big = 4096
        reps = -(-big // nvar)
        lens = np.diff(offs.astype(np.int64))
        offs_big = np.zeros(big + 1, dtype=np.uint64)
        offs_big[1:] = np.cumsum(np.tile(lens, reps)[:big])
        comp_big = torch.from_numpy(np.tile(comp, reps)[: int(offs_big[-1])].copy()).pin_memory().numpy()
        st_big = capi.Step2(X, mask, in_an, N, big)
        st_big.bgen_inflate(comp_big, offs_big, N)
        t0 = time.perf_counter()
        for _ in range(2):
            st_big.bgen_inflate(comp_big, offs_big, N)
        ti = (time.perf_counter() - t0) / 2
        st_big.close()
        inflate["direct_4096_streams_per_launch"] = {"inflate_ms_per_launch": 1e3 * ti, "inflated_GBps": big * (10 + 3 * N) / ti / 1e9,
                                                     "variants_per_sec_inflate_only": big / ti,
                                                     "note": "compressed bytes (pinned host) -> device, inflate kernel, payload split; no score test"}
    except Exception as e:
        inflate["direct_4096_streams_per_launch"] = {"error": str(e)[:200]}
    cpu = None
    if not args.no_cpu:
        thr = host_threads()
        reps = 16                                      # the 400 synthetic variants, 16 times over: a few seconds of CPU work
        nv_cpu = reps * nvar
        pm = np.full((nvar, N), 2, dtype=np.uint8)
        ref_eigen.s2_block_bt_probs(probs_np[:32], pm[:32], N, in_an, gsm, X, yres, threads=thr)
        t0 = time.perf_counter()
        for _ in range(reps):
            ref_eigen.s2_block_bt_probs(probs_np, pm, N, in_an, gsm, X, yres, threads=thr)
        dt = time.perf_counter() - t0
        cpu = {"value": nv_cpu / dt, "unit": "variants/s", "cores": thr, "kind": "port",
               "sample": "%d variants at N=%d: C++/Eigen restatement of the BGEN dosage loop + compute_score_bt (score statistic "
                         "only, no Firth, payloads already inflated), one OpenMP task per variant (%.2f s)" % (nv_cpu, N, dt)}
    return {"metric": "step2_bt_bgen_variants_per_sec", "value": dev_rate, "unit": "variants/s",
            "e2e": {"value": max(host_rate, staged_rate), "unit": "variants/s", "h2d_bytes_per_variant": 3 * N, "d2h_bytes_per_variant": 8 * 10 + 12,
                    "staged": staged_rate, "unstaged": host_rate},
            "e2e_compressed_input": inflate,
            "compressed_bytes_per_variant": float(offs[-1]) / nvar,
            "roofline": hbm_roofline(dev_rate, 3.0 * N, "2N probability bytes + N ploidy bytes",
                                     step2_traffic_from_profile(("dosage_relayout_kernel", "dosage_stats_kernel", "s2_bt_finalize_kernel"), 400)
                                     if N == 100_000 else (None, None)),
            "cpu_baseline": cpu, "firth_fraction": ff,
            "sample": "%d blocks of %d variants, N=%d, 1 binary trait (prevalence 10 %%), score test + approximate Firth for |z| > 1.96; "
                      "value = inflated bytes resident in HBM, e2e = pinned host probability + ploidy bytes (3N B/variant), "
                      "e2e_compressed_input = zlib payloads from host memory, inflated on the device (direct / shared-memory "
                      "window kernel) in front of the same calls" % (nblocks, nvar, N)}


def gram_traffic_from_profile():
    """DRAM bytes per launch and tensor-pipe activity of the Gram kernel from the committed ncu --set full summary
    (bench.py cannot run under a profiler; the capture command is tools/ncu_capture.sh)."""
    blocks = []
    for name in ("ncu_r2o_key_kernels.txt", "ncu_r1n_key_kernels.txt"):      # newest committed capture first
        try:
            blocks = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", name)).read().split("---\n")
            break
        except OSError:
            continue
    for b in blocks:
        if "gram_fp8_tcgen05_kernel" not in b or "launch__grid_size" not in b:
            continue
        d = {}
        for line in b.splitlines():
            t = line.split()
            if len(t) >= 2:
                d[t[0]] = t[1]
        if d.get("launch__grid_size") != "360":            # the bs x bs Gram launch (72 tiles x 5 folds), not the statistics tiles
            continue
        mb = float(d["dram__bytes_read.sum"]) + float(d["dram__bytes_write.sum"])
        return mb * 1e6, float(d["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"]) / 100.0
    return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--small", action="store_true", help="tiny config for smoke runs (not a bench value)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-step2", action="store_true")
    ap.add_argument("--cpu-blocks", type=int, default=1)
    ap.add_argument("--blocks", type=int, default=0, help="profiling only: restrict the pass to the first n blocks")
    ap.add_argument("--n-samples", type=int, default=0, help="exploration only: other sample count, --blocks blocks (default 20)")
    ap.add_argument("--n-pheno", type=int, default=0, help="exploration only: other trait count (configs[4] has 50)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the level-0 predictors of the last one (a fixed sample of rows) "
                         "to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs runs on one GPU (sharded, each rank holds the predictors of its own phenotypes only)")
    from oracle import ref_eigen
    if args.impl == "b200" and not args.no_cpu and not ref_eigen.available():
        sys.stderr.write("bench.py: oracle/_ref/libregenie_ref_eigen*.so not built (it needs the reference's sources): "
                         "running without the CPU baseline and its parity check\n")
        args.no_cpu = True
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
