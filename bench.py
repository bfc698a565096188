#!/usr/bin/env python3
"""bench.py -- MarlinKZG10/BLS12-381 commit+open at degree 2^20 (BASELINE.json configs[1]) on N B200s.

A step = one KZG10 commit + one KZG10 open of one degree-2^20 polynomial (2^20+1 uniform Fr coefficients,
hiding_bound=None, degree_bound=None: the protocol of bench-templates/src/lib.rs:69-138) = two G1 MSMs of
2^20(+1) terms, one division by (X - z), with F::into_bigint fused into the MSM digit pass.

  value   whole-job polys/s with the coefficient vectors already resident in HBM (PCGPU_DEVICE_PTRS)
  e2e     the same through the C ABI with pinned HOST buffers (H2D of the coefficients inside the timed region,
          D2H of the two 96-byte points)
  roofline    dominant kernel (round 0 of the batched-affine pair rounds): algorithmic bytes (128 B per scalar-mult, SURVEY.md 8d) over the
              average launch duration from CUDA events on the launching stream; peak = MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle port (oracle/, OpenMP over Pippenger windows) timed on this box's host cores
  --impl reference   times that CPU path alone (the reference's Rust cannot be built here: no cargo/rustc)

Multi-GPU: ranks shard by polynomial (SURVEY.md 8e partitioning A; the reference's per-polynomial loop,
marlin_pc/mod.rs:192), SRS replicated, no data-path collective; weak scaling.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

LOG_DEG = 20
CURVE = "bls12_381"
ALGO_BYTES_PER_SCALAR_MULT = 128  # 96 B affine base + 32 B scalar (SURVEY.md section 8d)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="pcgpu", choices=["pcgpu", "reference"])
    ap.add_argument("--log-deg", type=int, default=LOG_DEG)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the sharded MSM / cfg5 / NTT sub-record")
    ap.add_argument("--sharded-log-n", type=int, default=22)
    ap.add_argument("--cfg5-polys", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the commitment and witness of the last timed step to DIR/<name>.npy "
                         "(float64; each 64-bit Montgomery limb of x||y as two 32-bit words, low word first)")
    return ap.parse_args()


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,"
         "timestamp")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        """start of the timed region: only samples taken after this moment are reported"""
        import datetime
        self.t_mark = datetime.datetime.now()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        import datetime
        rows = []
        for r in self.rows:
            if len(r) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(r[9], "%Y/%m/%d %H:%M:%S.%f")
            except Exception:
                continue
            if getattr(self, "t_mark", None) is None or ts >= self.t_mark:
                rows.append(r)
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in rows for k in range(4) if r[5 + k].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_threads():
    """threads the CPU arm may use: every core this process is allowed on (torchrun exports OMP_NUM_THREADS=1, which
    would otherwise cripple the OpenMP default)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def oracle_step(orc, cid, bases, coeffs, z, nthreads=0):
    rc, cxy, cinf = orc.kzg_commit(cid, bases, coeffs, nthreads=nthreads)
    assert rc == 0
    rc, wxy, winf, _ = orc.kzg_open(cid, bases, coeffs, z, nthreads=nthreads)
    assert rc == 0
    return cxy, wxy


def pippenger_ops(n):
    """point additions of the oracle's Pippenger (ark-ec window rule) for an n-term 255-bit MSM."""
    import math
    c = 3 if n < 32 else int(math.log2(n)) * 69 // 100 + 2
    w = (255 + c - 1) // c
    return w * (n + 2 * ((1 << c) - 1))


def cpu_reference_run(args, log_deg, steps, warmup, budget_s):
    """The CPU path (oracle port of the reference's dataflow; OpenMP across windows like ark-ec's Rayon MSM)."""
    import numpy as np
    from oracle import orc, pyref
    from tests import util
    C = pyref.Curve(CURVE)
    n_full = (1 << log_deg) + 1
    import math
    c_win = 3 if n_full < 32 else int(math.log2(n_full)) * 69 // 100 + 2
    n_windows = (255 + c_win - 1) // c_win
    # like ark-ec's Rayon MSM the port parallelises over Pippenger windows only, so at most n_windows threads do work
    # (splitting the index range as well was tried: 8 slices x 17 windows on the 128-thread box ran 2x SLOWER -- every
    # slice pays its own 2^c-bucket reduction and the bucket arrays fall out of cache)
    cores = min(host_threads(), n_windows)
    # SRS for the CPU run: random multiples of G (fixed-base batch mul on the host is the slow part, so the
    # base set is 2^14 distinct points tiled -- MSM cost does not depend on the base values)
    tile = 1 << 14
    pts = util.random_points(CURVE, tile, seed=99)
    z = util.rand_fr(CURVE, 1, seed=4, mont=True)[0]

    def run(n):
        reps = (n + tile - 1) // tile
        bases = np.tile(pts, (reps, 1))[:n]
        coeffs = util.rand_fr_fast(CURVE, n, 7)
        t0 = time.perf_counter()
        oracle_step(orc, C.id, bases, coeffs, z, nthreads=host_threads())
        return time.perf_counter() - t0

    # probe at 1/16 size to choose the sample
    t_probe = run((1 << max(log_deg - 4, 8)) + 1)
    est_full = t_probe * pippenger_ops(n_full) / pippenger_ops((1 << max(log_deg - 4, 8)) + 1)
    if est_full * (steps + warmup) <= budget_s:
        n_s, scale, sample = n_full, 1.0, f"full workload: commit+open of one degree-2^{log_deg} polynomial per step"
    else:
        shift = 2
        while shift < 8 and est_full / (1 << shift) * (steps + warmup) > budget_s:
            shift += 1
        n_s = (1 << (log_deg - shift)) + 1
        scale = pippenger_ops(n_full) / pippenger_ops(n_s)
        sample = (f"commit+open of a degree-2^{log_deg - shift} polynomial per step, time scaled x{scale:.2f} by the "
                  f"Pippenger point-addition count to degree 2^{log_deg}")
    for _ in range(warmup):
        run(n_s)
    times = [run(n_s) for _ in range(steps)]
    t = sum(times) / len(times) * scale
    sample += f"; OpenMP over the {n_windows} Pippenger windows ({host_threads()} host threads available)"
    return {"value": 1.0 / t, "unit": "polys/s", "cores": cores, "kind": "port", "sample": sample,
            "ms_per_step": t * 1e3, "msm_scalar_mults_per_s": 2 * n_full / t}


def dump_outputs(out_dir, c, ci, w, wi):
    """the arrays the batch call returns for one polynomial, exactly: 64-bit limbs split into 32-bit words fit float64"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    words = lambda xy: np.ascontiguousarray(xy, dtype=np.uint64).view(np.uint32).astype(np.float64)
    for name, a in (("commitment_xy", words(c)), ("commitment_inf", np.float64([ci])),
                    ("witness_xy", words(w)), ("witness_inf", np.float64([wi]))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    log_deg = args.log_deg
    workload = f"MarlinKZG10 commit+open, 1 poly/step, degree 2^{log_deg}, BLS12-381, hiding_bound=None, degree_bound=None"

    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps if args.steps is not None else 3
        warmup = args.warmup if args.warmup is not None else 1
        r = cpu_reference_run(args, log_deg, steps, warmup, budget_s=float(os.environ.get("PCGPU_REF_BUDGET_S", "200")))
        line = {"impl": "reference", "metric": "MarlinKZG10/BLS12-381 commit+open polys/s at deg 2^20", "value": r["value"],
                "unit": "polys/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64-limb Montgomery (CPU)",
                "data": "synthetic", "config": {"workload": workload, "reference": "CPU oracle port of the reference dataflow "
                "(ark-ec/ark-poly cannot be built here: no Rust toolchain)"},
                "msm_scalar_mults_per_s": r["msm_scalar_mults_per_s"],
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": "polys/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    steps = args.steps if args.steps is not None else 20
    warmup = args.warmup if args.warmup is not None else 3
    import numpy as np
    import torch
    import pkgload
    pc = pkgload.load()
    from poly_commit_b200 import params, sharded  # the oracle is imported by the cpu_baseline leg only (cpu_reference_run)

    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        dist = SingleDist()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    eng = pc.Engine(local_rank)  # raises without the CUDA library / an sm_100 device
    cid = pc.CURVES[CURVE]
    n = (1 << log_deg) + 1

    # ---- synthetic SRS on the device: P_i = k_i G for seeded random k_i (g.batch_mul, kzg10/mod.rs:76, with random
    # scalars in place of the powers of beta: the commit / open kernels do not depend on the structure of the bases), then
    # window-folded tables
    pows = torch.from_numpy(params.random_fr(cid, n, 1001).view(np.int64)).cuda()
    d_bases = torch.empty((n, 12), dtype=torch.int64, device="cuda")
    eng.fixed_base_mul(cid, params.g1_generator(cid), pows.data_ptr(), n=n, flags=pc.DEVICE_PTRS, out=d_bases.data_ptr())
    srs = eng.srs_register(cid, d_bases.data_ptr(), n=n, flags=pc.DEVICE_PTRS | pc.SRS_PRECOMPUTE)
    del pows

    # ---- polynomials: distinct per rank and per step (rotating), pinned host copies + device copies
    n_polys = 4
    host_polys = [torch.from_numpy(params.random_fr(cid, n, 100 + rank * n_polys + i).view(np.int64)).pin_memory() for i in range(n_polys)]
    dev_polys = [h.cuda() for h in host_polys]
    host_views = [h.numpy().view(np.uint64) for h in host_polys]
    z = params.random_fr(cid, 1, 4)[0]

    # One step = commit + open of one polynomial.  The timed region is ONE call of the library's batch entry point over the
    # K polynomials of the K steps (pcgpu_kzg_commit_open_batch: coefficients uploaded once per polynomial, two polynomials in
    # flight, each with its commitment and witness MSM pipelines on two streams) -- a single host thread, no Python threading.
    def run_dev(k):
        return eng.kzg_commit_open_batch(srs, [(dev_polys[i % n_polys].data_ptr(), n) for i in range(k)], z, flags=pc.DEVICE_PTRS)

    def run_host(k):
        return eng.kzg_commit_open_batch(srs, [host_views[i % n_polys] for i in range(k)], z)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # the library's calls are synchronous (each ends with a sync of its own streams), so events recorded on the
        # current stream before the call and after it bracket all the work of all its streams
        e0.record()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = fn(k)
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        e1.record()
        torch.cuda.synchronize()
        ms = max(e0.elapsed_time(e1), wall_ms)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, res

    sampler = ClockSampler(local_rank)
    sampler.start()                      # started before the warm-up so nvidia-smi is already streaming samples
    run_dev(max(warmup, 3))
    sampler.mark()
    l0 = eng.launch_count()
    ms_dev, (c, ci, w, wi) = timed(run_dev, steps)
    launches = eng.launch_count() - l0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, c[-1], ci[-1], w[-1], wi[-1])
    run_host(max(warmup, 3))
    ms_host, _ = timed(run_host, steps)
    # single-call latency (one polynomial per call: what a serial Rust caller of commit-then-open sees)
    eng.kzg_commit_open(srs, dev_polys[0].data_ptr(), z, n=n, flags=pc.DEVICE_PTRS)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(min(steps, 8)):
        eng.kzg_commit_open(srs, dev_polys[i % n_polys].data_ptr(), z, n=n, flags=pc.DEVICE_PTRS)
    torch.cuda.synchronize()
    ms_single_call = (time.perf_counter() - t0) * 1e3 / min(steps, 8)
    # kernel-level timings: a separate pass with ONE pipeline in flight (commit, then open), CUDA events around every stage
    # on the launching stream (with several pipelines in flight the per-stage times would include the other pipeline's kernels)
    eng.profile_enable(True)
    prof_steps = min(steps, 8)
    for i in range(prof_steps):
        d = dev_polys[i % n_polys]
        eng.kzg_commit(srs, d.data_ptr(), n=n, flags=pc.DEVICE_PTRS)
        eng.kzg_open(srs, d.data_ptr(), z, n=n, flags=pc.DEVICE_PTRS)
    acc_ms, acc_cnt = eng.profile_get(4)
    stage_ms = {name: eng.profile_get(s)[0] / max(prof_steps, 1) for s, name in
                enumerate(["digits_count", "scan", "scatter", "tasks", "bucket_accumulate", "bucket_reduce", "final_host", "fr_division"])}
    stage_ms["affine_pair_rounds"] = eng.profile_get(11)[0] / max(prof_steps, 1)
    pair0_ms, pair0_cnt = eng.profile_get(12)
    eng.profile_enable(False)

    shard = None
    if not args.no_sharded:
        try:
            shard = sharded_record(args, eng, pc, params, sharded, dist, dev, rank, world, cid)
        except Exception as e:  # the headline line must survive a failure of the extra record
            shard = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    polys = steps * world
    value = polys / (ms_dev / 1e3)
    e2e = polys / (ms_host / 1e3)
    peak, peak_src = measured_peaks()
    # compute roofline that actually binds the MSM: wide integer multiply-adds per second (measured live on this GPU)
    imad_peak = eng.measure_imad_peak()
    # multiply count of one 2^log_deg MSM: entries = n * W windows, 3 affine rounds at 6.2 modmuls, the rest XYZZ at 9.5,
    # 288 wide multiplies per 12-limb Montgomery product
    windows = 15 if log_deg >= 18 else 16
    msm_entries = n * windows
    wide_per_msm = (msm_entries * (7.0 / 8.0) * 6.2 + msm_entries * (1.0 / 8.0) * 9.5) * 288
    msm_kernel_ms = (stage_ms["affine_pair_rounds"] + stage_ms["bucket_accumulate"]) / 2
    # dominant kernel = round 0 of the batched-affine pair rounds (one launch per MSM, touches every (base, scalar) pair)
    dom_ms = pair0_ms / pair0_cnt if pair0_cnt else (acc_ms / max(acc_cnt, 1))
    dom_name = "run_kernel_occ<MsmAffinePairBody<Bls12381, true>>" if pair0_cnt else "run_persistent_kernel<MsmAccumulateBody<Bls12381>>"
    achieved = (n * ALGO_BYTES_PER_SCALAR_MULT / 1e9) / (dom_ms / 1e3) if dom_ms else None
    traffic, traffic_src = ncu_traffic(log_deg)
    line = {
        "metric": "MarlinKZG10/BLS12-381 commit+open polys/s at deg 2^20", "value": value, "unit": "polys/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_dev / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32-limb Montgomery (Fq 381-bit x12, Fr 255-bit x8)",
        "data": "synthetic",
        "config": {"workload": workload, "parallelism": f"poly-sharded x{world}, SRS replicated; one batch call per rank, 2 polynomials "
                   "(4 MSM pipelines) in flight inside the library",
                   "l2": "per-step working set (window-folded SRS tables 1.5 GB gather + 34 MB coefficients, rotating "
                         "polynomials) exceeds the 126 MB L2; no explicit flush"},
        "msm_scalar_mults_per_s": 2 * n * polys / (ms_dev / 1e3),
        "stage_ms_per_step": stage_ms,
        "single_call_ms_per_step": ms_single_call,
        "e2e": {"value": e2e, "unit": "polys/s", "h2d_bytes_per_step": n * 32 + 32, "d2h_bytes_per_step": 2 * 96 + 2 * 4,
                "ms_per_step": ms_host / steps},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src, "launch_ms": dom_ms,
                     "compute_roofline": {"bound": "int32 multiply pipe (IMAD.WIDE.U32)", "peak_wide_mul_per_s": imad_peak,
                                          "achieved_wide_mul_per_s": wide_per_msm / (msm_kernel_ms / 1e3) if msm_kernel_ms else None,
                                          "frac": (wide_per_msm / (msm_kernel_ms / 1e3) / imad_peak) if (msm_kernel_ms and imad_peak) else None,
                                          "kernels": "pair rounds x3 + MsmAccumulateBody, per MSM (multiply counts assumed: 6.2 / 9.5 modmuls "
                                                     "per affine / XYZZ addition, 288 wide multiplies per modmul)"},
                     "note": "MSM is INT32-multiply bound (~3.4k IMAD.WIDE per 128 algorithmic bytes); the HBM fraction "
                             "is reported because north_star asks for it"},
    }
    if shard is not None:
        line["sharded"] = shard
    if not args.no_cpu_baseline and world == 1:
        cb = cpu_reference_run(args, log_deg, steps=1, warmup=0, budget_s=25.0)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


class SingleDist:
    """the torch.distributed calls the sharded helpers use, for a world of one process (python bench.py --gpus 1)"""

    class ReduceOp:
        MAX = "max"
        MIN = "min"

    def get_rank(self):
        return 0

    def get_world_size(self):
        return 1

    def barrier(self):
        pass

    def all_gather(self, outs, t):
        outs[0].copy_(t)

    def all_reduce(self, t, op=None):
        return t

    def all_to_all_single(self, out, inp):
        out.copy_(inp)


def ncu_traffic(log_deg):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the committed ncu --set full
    capture of THIS code (profiles/r02_ncu_pair0_traffic.json, written by tools/ncu_traffic.py from the capture's raw page)"""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_pair0_traffic.json")) as f:
            d = json.load(f)
        if int(d.get("log_deg", -1)) == log_deg:
            return int(d["dram_bytes_read"]) + int(d["dram_bytes_write"]), d.get("source")
    except Exception:
        pass
    return None, None


def sharded_record(args, eng, pc, params, sharded, dist, dev, rank, world, cid):
    """The north_star's multi-GPU splits, measured next to the headline (same process group, device-resident, max over ranks):
      msm        ONE 2^22-term MSM sharded by index range over the N GPUs: fused NVLink point-sum (pcgpu_msm_peer), the NCCL
                 all-gather baseline, and the same MSM on one GPU (every rank runs it; the slowest rank is reported)
      cfg5       BASELINE.json configs[4]: 64 polynomials of degree 2^22 committed over the N GPUs (sharded by polynomial,
                 SRS replicated), commitments gathered with NCCL
      ntt        one 2^22 NTT sharded by the four-step split: exchange fused into pass 1 (NVLink stores + flag barrier), the NCCL
                 all-to-all baseline, and the single-GPU transform"""
    import numpy as np
    import torch
    log_n = args.sharded_log_n
    n = (1 << log_n) + 1
    out = {"log_n": log_n}

    def tmax(fn, reps):
        torch.cuda.synchronize(dev); dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize(dev)
        dt = (time.perf_counter() - t0) / reps * 1e3
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt

    ks = torch.from_numpy(params.random_fr(cid, n, 2001).view(np.int64)).to(dev)
    d_bases = torch.empty((n, 12), dtype=torch.int64, device=dev)
    eng.fixed_base_mul(cid, params.g1_generator(cid), ks.data_ptr(), n=n, flags=pc.DEVICE_PTRS, out=d_bases.data_ptr())
    del ks
    full = eng.srs_register(cid, d_bases.data_ptr(), n=n, flags=pc.DEVICE_PTRS | pc.SRS_PRECOMPUTE)
    base_polys = [torch.from_numpy(params.random_fr(cid, n, 3000 + i).view(np.int64)).to(dev) for i in range(2)]
    fl = pc.SCALARS_MONT | pc.DEVICE_PTRS
    peers = sharded.PeerGroup(eng, dist, device=dev if world > 1 else None)
    # ---- one MSM, index-sharded
    d_sc = base_polys[0]
    ref = eng.msm(full, d_sc.data_ptr(), n=n, flags=fl)
    single_ms = tmax(lambda: eng.msm(full, d_sc.data_ptr(), n=n, flags=fl), 3)
    res = {}
    for mode in ("peer", "nccl"):
        if world == 1:
            sm_srs_owner = None
        sm = sharded.ShardedMsm(eng, cid, d_bases.data_ptr(), dist, flags=pc.SRS_PRECOMPUTE, device=dev if world > 1 else None, n=n,
                                peers=peers if mode == "peer" else None, mode=mode)
        lo, hi = sm.local_slice()
        ptr = d_sc.data_ptr() + lo * 32
        got = sm.msm(ptr, flags=fl, n=n)
        res[mode + "_ok"] = bool((got[0] == ref[0]).all() and got[1] == ref[1])
        res[mode + "_ms"] = tmax(lambda: sm.msm(ptr, flags=fl, n=n), 3)
        sm.srs.release()
    out["msm"] = {"terms": n, "single_gpu_ms": round(single_ms, 3), "sharded_nvlink_fused_ms": round(res["peer_ms"], 3),
                  "sharded_nccl_allgather_ms": round(res["nccl_ms"], 3), "bit_exact_vs_single_gpu": res["peer_ok"] and res["nccl_ok"],
                  "scalar_mults_per_s": round(n / (res["peer_ms"] / 1e3)), "speedup_vs_single_gpu": round(single_ms / res["peer_ms"], 3),
                  "collective": f"{world} x ~3.3 KB bit-plane records stored into the peers' windows by the pipeline's last kernel, "
                                "flag wait, one D2H copy; bounded by the slowest rank's Pippenger pipeline, not by the exchange"}
    # ---- cfg5: 64 polynomials over the ranks
    npoly = args.cfg5_polys
    mine = sharded.poly_assignment(npoly, rank, world)
    polys = []
    for i in mine:   # distinct polynomials derived on the device: p_i = base_0 * c_i + base_1
        p = base_polys[1].clone()
        eng.fr_axpy(cid, p.data_ptr(), params.random_fr(cid, 1, 4000 + i)[0], base_polys[0].data_ptr(), n=n, flags=pc.DEVICE_PTRS)
        polys.append(p)
    torch.cuda.synchronize(dev)
    run = lambda: sharded.commit_batch_sharded(eng, full, [(p.data_ptr(), n) for p in polys], dist, device=dev if world > 1 else None,
                                               flags=pc.DEVICE_PTRS, num_polys=npoly)
    comms, _ = run()
    spot = eng.kzg_commit(full, polys[0].data_ptr(), n=n, flags=pc.DEVICE_PTRS)
    ms = tmax(run, 1)
    out["cfg5"] = {"workload": f"Batched MarlinKZG10 commit, {npoly} polys, degree 2^{log_n}, BLS12-381, sharded by polynomial over {world} GPU(s)",
                   "ms_total": round(ms, 2), "polys_per_s": round(npoly / (ms / 1e3), 2), "scalar_mults_per_s": round(npoly * n / (ms / 1e3)),
                   "spot_check_ok": bool((comms[mine[0]] == spot[0]).all()),
                   "collective": "NCCL all_gather of the commitments (104 bytes per polynomial) after the local batches; no data-path exchange"}
    del polys
    full.release()
    del d_bases
    torch.cuda.empty_cache()
    # ---- one NTT, four-step sharded
    ntt_log = min(log_n, 22)
    n_in = (1 << ntt_log) - 3
    x = base_polys[0]
    exp = torch.empty((1 << ntt_log, 4), dtype=torch.int64, device=dev)
    eng.ntt(cid, x.data_ptr(), ntt_log, n_in=n_in, flags=pc.DEVICE_PTRS, out=exp.data_ptr())
    ntt_single = tmax(lambda: eng.ntt(cid, x.data_ptr(), ntt_log, n_in=n_in, flags=pc.DEVICE_PTRS, out=exp.data_ptr()), 5)
    rec = {"log_n": ntt_log, "single_gpu_ms": round(ntt_single, 4)}
    m1, m2 = eng.ntt_split(ntt_log)
    if world > 1 and (1 << m1) % world == 0 and (1 << m2) % world == 0:
        pn = sharded.PeerNtt.from_group(eng, cid, ntt_log, peers)
        rows = pn.N1 // world
        o1 = torch.empty((pn.N2, rows, 4), dtype=torch.int64, device=dev)
        pn.forward_rank(x.data_ptr(), n_in, o1.data_ptr())
        want = exp.view(pn.N2, pn.N1, 4)[:, rank * rows:(rank + 1) * rows, :]
        ok = bool((o1 == want).all())
        rec["sharded_nvlink_fused_ms"] = round(tmax(lambda: pn.forward_rank(x.data_ptr(), n_in, o1.data_ptr()), 5), 4)
        sn = sharded.ShardedNtt(eng, cid, ntt_log, dist, device=dev)
        ok = ok and bool((sn.forward_device(x, n_in) == want).all())
        rec["sharded_nccl_alltoall_ms"] = round(tmax(lambda: sn.forward_device(x, n_in), 5), 4)
        okt = torch.tensor([int(ok)], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        rec["bit_exact_vs_single_gpu"] = bool(okt.item())
        rec["speedup_vs_single_gpu"] = round(ntt_single / rec["sharded_nvlink_fused_ms"], 3)
        rec["nvlink_bytes_per_rank"] = (1 << ntt_log) * 32 * (world - 1) // (world * world)
        rec["collective"] = "pass-1 blocks store their outputs straight into the row owners' buffers (NVLink P2P), epoch-flag barrier, pass 2"
    out["ntt"] = rec
    peers.close()
    return out


if __name__ == "__main__":
    main()
