#!/usr/bin/env python
"""bench.py -- headline benchmark of the MSM / NTT hot paths.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--lg-msm 26] [--lg-ntt 24]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one BLS12-381 G1 MSM over 2^26 synthetic points (BASELINE.json's headline metric),
sharded by point-chunk over the N ranks with one all-gather of the per-rank partial results
(strong scaling: the MSM size is fixed).  `value` is device-resident throughput, `e2e` goes
through the drop-in C-ABI `mult_pippenger` with HOST (pinned) buffers (at N > 1: every rank's
shard through `mult_pippenger`, then the same all-gather + combine).  The Goldilocks 2^24 NTT
(the metric's second half) is measured in the same run and reported under "ntt".
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over
ranks.  Inputs (8.6 GB MSM, 2 x 128 MiB NTT + L2 flush) exceed the 126 MB L2.  Every timed
loop of every leg runs exactly --steps iterations; the untimed warm-up runs --warmup of them
(at least 3 for the NTT and Pallas legs, whose first calls build tables and pools).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

R_BLS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
GL_P = 2**64 - 2**32 + 1
LG_DISTINCT = 16            # distinct points, replicated (the reference's util.rs replicates 2^11)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled every 10 ms from
    a thread (a short multi-GPU run lasts less than one nvidia-smi start-up); nvidia-smi -lms as
    the fallback when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.nvml, self.h, self.stop_flag, self.samples, self.mask, self.max = None, None, False, [], 0, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                fn = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
                self.mask |= int(fn(self.h))
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
            sm = sorted(self.samples)
            busy = [v for v in sm if v > 0.5 * (self.max or 1)] or sm
            return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": self.max,
                    "reasons": sorted(nm for bit, nm in self.BITS.items() if self.mask & bit),
                    "samples": len(sm), "source": "nvml, 10 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 4 + k and r[4 + k].lower().startswith("active"):
                    reasons.add(nm)
        busy = [v for v in sm if v > 0.5 * (mx[0] if mx else 1)] or sm
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 200"}


def fold_scalars(sc, m, r=None):
    """sum of scalars per residue class i mod m, reduced mod r -> (m, 4) uint64."""
    r = R_BLS if r is None else r
    n = sc.shape[0]
    v = sc.reshape(n // m, m, 4)
    lo = (v & np.uint64(0xFFFFFFFF)).sum(axis=0, dtype=np.uint64)       # < 2^32 * n/m
    hi = (v >> np.uint64(32)).sum(axis=0, dtype=np.uint64)
    out = np.zeros((m, 4), dtype=np.uint64)
    for j in range(m):
        t = 0
        for k in range(4):
            t += (int(lo[j, k]) + (int(hi[j, k]) << 32)) << (64 * k)
        t %= r
        for k in range(4):
            out[j, k] = (t >> (64 * k)) & 0xFFFFFFFFFFFFFFFF
    return out


def cpu_reference_msm(points, scalars, nthreads):
    """sppark's CPU path on the host cores: the reference's own msm/pippenger.hpp when oracle/_ref
    holds it (built in the authoring container from /root/reference), else the C restatement."""
    from oracle import pyoracle
    t0 = time.perf_counter()
    if pyoracle.ref_cpu() is not None:
        out = pyoracle.ref_cpu_msm(points, scalars, nthreads=nthreads)
        kind = "reference"
    else:
        out = pyoracle.msm("bls12_381", points, scalars, "pippenger", ncpus=nthreads)
        kind = "port"
    return out, time.perf_counter() - t0, kind


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on this box's cores."""
    if rank != 0:
        return
    from oracle import pyoracle          # the reference arm runs no kernel of this repository
    lg_s = args.lg_cpu_sample
    n = 1 << lg_s
    cores = os.cpu_count() or 1
    base = pyoracle.gen_points("bls12_381", 1 << min(12, lg_s))
    pts = np.tile(base, (n // base.shape[0], 1))
    rng = np.random.default_rng(1234)
    sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
    sc[:, 3] >>= np.uint64(2)
    for _ in range(args.warmup):
        cpu_reference_msm(pts[: n // 8], sc[: n // 8], cores)
    t = 0.0
    kind = "port"
    for _ in range(args.steps):
        _, dt, kind = cpu_reference_msm(pts, sc, cores)
        t += dt
    per_step = t / args.steps
    value = (n / per_step) / (1 << args.lg_msm)        # MSM/s at 2^lg_msm points, by point throughput
    sample = (f"2^{lg_s}-point MSM per step on {cores} host threads; value = points/s / 2^{args.lg_msm} "
              "(Pippenger cost per point falls slowly with size, so this slightly under-estimates 2^26)")
    line = {"impl": "reference", "metric": f"BLS12-381 G1 MSM/s @2^{args.lg_msm} points", "value": value,
            "unit": "MSM/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64x6 Montgomery (portable, no blst asm)", "data": "synthetic",
            "config": {"workload": f"bls12_381_g1_msm_2^{args.lg_msm}", "cpu_sample": f"2^{lg_s}"},
            "cpu_baseline": {"value": value, "unit": "MSM/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "MSM/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


_JSON_OUT = None


def emit(line):
    """The one JSON line, on the process's ORIGINAL stdout."""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout carries exactly one JSON line: anything a library prints on fd 1 (NCCL's version
    # banner, for one) is sent to stderr instead
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--lg-msm", type=int, default=26)
    ap.add_argument("--lg-ntt", type=int, default=24)
    ap.add_argument("--lg-cpu-sample", type=int, default=22)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-ref-gpu", action="store_true")
    ap.add_argument("--lg-pallas", type=int, default=24)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of each leg returned to DIR/<name>.npy "
                         "(float64, every value exact; see dump_outputs).  With one rank: the BLS12-381 and Pallas "
                         "MSMs and the Goldilocks NTT; with several ranks: the two MSMs only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":            # CPU only: no CUDA, no process group
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from sppark_b200 import _lib, msm, ntt

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------------------------------------------------------- synthetic MSM shard
    n_total = 1 << args.lg_msm
    n = n_total // world
    m = 1 << min(LG_DISTINCT, args.lg_msm - (world.bit_length() - 1))
    base_dev = msm.generate_points_dev(msm.BLS12_381_G1, m)
    torch.cuda.synchronize()
    base = base_dev.cpu().numpy().view(np.uint64)                     # (m, 12)
    rng = np.random.default_rng(42 + rank)
    need_host = not args.skip_e2e and world == 1
    if need_host:
        pts_host_t = torch.empty((n, 12), dtype=torch.int64, pin_memory=True)
        sc_host_t = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
        pts_host, sc_host = pts_host_t.numpy().view(np.uint64), sc_host_t.numpy().view(np.uint64)
    else:
        sc_host = np.empty((n, 4), dtype=np.uint64)
    blk = 1 << 22
    for s in range(0, n, blk):
        e = min(n, s + blk)
        sc_host[s:e] = rng.integers(0, 2**64, size=(e - s, 4), dtype=np.uint64)
    sc_host[:, 3] >>= np.uint64(2)                                     # uniform below 2^254 < r
    d_points = base_dev.repeat(n // m, 1).contiguous()
    d_scalars = torch.from_numpy(sc_host.view(np.int64)).cuda()
    if need_host:
        pts_host.reshape(n // m, m, 12)[:] = base
    torch.cuda.synchronize()

    from sppark_b200 import parallel

    def msm_step():
        # local chunk -> one Jacobian point; all-gather of 144 B per rank (NCCL over NVLink);
        # the partials are added on the GPU by the library (sppark_b200_msm_combine)
        return parallel.msm_sharded(lambda: msm.msm_dev(msm.BLS12_381_G1, d_points, d_scalars),
                                    lambda parts: msm.combine(msm.BLS12_381_G1, parts) if world > 1 else parts[0],
                                    18, device="cuda")

    launches0 = _lib.launch_count()
    for _ in range(args.warmup):
        result = msm_step()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    launches1 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        result = msm_step()
    e1.record()
    barrier()
    clocks = sampler.stop()
    gpu_launches = _lib.launch_count() - launches1
    ms_step = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    value = 1e3 / ms_step

    # ---- roofline leg: the dominant kernel (bucket accumulation), timed live with CUDA events
    _lib.profile_enable(True)
    acc_ms = []
    for _ in range(args.steps):
        msm.msm_dev(msm.BLS12_381_G1, d_points, d_scalars)
        phases = dict(_lib.profile_read())
        acc_ms.append(phases.get("accumulate", 0.0))
    _lib.profile_enable(False)
    phases = {k: round(v, 3) for k, v in phases.items()}
    peak, peak_src = measured_peaks()
    alg_bytes = n * 128                              # 96-B affine point + 32-B scalar, read once
    acc = sum(acc_ms) / len(acc_ms)
    achieved = alg_bytes / (acc * 1e-3) / 1e9 if acc > 0 else 0.0
    # DRAM traffic of this kernel at 2^26 / c=20 from the committed `ncu --set full` capture
    # (profiles/msm_accumulate_r01.md: dram__bytes_read.sum + dram__bytes_write.sum per launch);
    # every point is gathered once per window, hence ~19x the algorithmic bytes
    traffic = 174.7e9 if (args.lg_msm == 26 and world == 1) else None      # profiles/msm_accumulate_r01.md (kernel unchanged)
    wide_mults = 2880.0 * phases_entries(n, world)          # 10 products x 288 IMAD.WIDE per mixed add
    imad_peak = 0.94 * 32 * 148 * 1.965e9                   # measured: tools/imad_bench.cu on this B200
    roofline = {"bound": "hbm", "kernel": "msm::accumulate_kernel", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms": acc, "phases_ms": phases,
                "int32_issue": {"achieved_wide_mults_per_s": wide_mults / (acc * 1e-3) if acc > 0 else 0.0,
                                "peak_wide_mults_per_s": imad_peak,
                                "frac": (wide_mults / (acc * 1e-3) / imad_peak) if acc > 0 else 0.0,
                                "note": "IMAD.WIDE.U32 issues at 0.94 warp-instr/clk/SM (tools/imad_bench.cu)"},
                "note": "bucket accumulation is bounded by INT32 multiply issue, not HBM; the HBM fraction is "
                        "reported because the contract asks for it (DESIGN.md section 5)"}

    # ---- self-check at full size (size-independent property, no oracle): folding the scalars of
    # the replicated points onto the m distinct points must give the same group element
    folded = fold_scalars(sc_host, m)
    if world > 1:
        # every rank holds the same m distinct points: the sharded MSM equals the m-point MSM whose
        # scalars are the folded scalars of ALL ranks, summed mod r
        parts = parallel.all_gather_partials(folded.reshape(-1), "cuda").reshape(world, m, 4)
        folded = fold_scalars(np.ascontiguousarray(parts.reshape(world * m, 4)), m)
    small = msm.msm_dev(msm.BLS12_381_G1, base_dev, torch.from_numpy(folded.view(np.int64)).cuda())
    check = f"folded-msm over {world} rank(s) " + ("ok" if _jac_equal(result, small, msm) else "MISMATCH")

    # ---------------------------------------------------------------- e2e through the C-ABI
    e2e = None
    if need_host:
        del d_points, d_scalars
        torch.cuda.empty_cache()
        msm.multi_scalar_mult(pts_host, sc_host)                        # warm the pools
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r2 = msm.multi_scalar_mult(pts_host, sc_host)
        dt = (time.perf_counter() - t0) / args.steps
        e2e = {"value": 1.0 / dt, "unit": "MSM/s", "h2d_bytes_per_step": int(n * 128),
               "d2h_bytes_per_step": 144, "ms_per_step": dt * 1e3, "api": "mult_pippenger (host pointers, pinned)",
               "same_result": bool(_jac_equal(r2, result, msm))}
        e2e_result = r2
    elif world > 1 and not args.skip_e2e:
        # N > 1: every rank pushes its shard through mult_pippenger from pinned host buffers (its
        # own PCIe link), then the same all-gather + combine as the device-resident step.  All
        # local work sits inside try/except and every rank ALWAYS joins the collectives, so one
        # rank's failure cannot leave the others waiting.
        failed = None
        try:
            pts_host_t = torch.empty((n, 12), dtype=torch.int64, pin_memory=True)
            pts_host_t.copy_(d_points)
            sc_host_t = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
            sc_host_t.copy_(d_scalars)
            torch.cuda.synchronize()
            pts_e2e, sc_e2e = pts_host_t.numpy().view(np.uint64), sc_host_t.numpy().view(np.uint64)
            del d_points, d_scalars
            torch.cuda.empty_cache()
        except Exception as e:
            failed = f"{type(e).__name__}: {e}"

        def local_host_msm():
            nonlocal failed
            if failed is None:
                try:
                    return msm.multi_scalar_mult(pts_e2e, sc_e2e)
                except Exception as e:
                    failed = f"{type(e).__name__}: {e}"
            return np.zeros(18, dtype=np.uint64)

        def e2e_step():
            return parallel.msm_sharded(local_host_msm, lambda parts: msm.combine(msm.BLS12_381_G1, parts), 18, device="cuda")

        e2e_step()                                                   # warm the pools
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r2 = e2e_step()
        barrier()
        dt = max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps) * 1e-3
        bad = max_over_ranks(0.0 if failed is None else 1.0)        # agreed on by all ranks
        if bad == 0.0:
            e2e = {"value": 1.0 / dt, "unit": "MSM/s", "h2d_bytes_per_step": int(n_total * 128),
                   "d2h_bytes_per_step": 144 * world, "ms_per_step": dt * 1e3,
                   "api": f"mult_pippenger on every rank's shard (host pointers, pinned), all-gather + combine; x{world}",
                   "same_result": bool(_jac_equal(r2, result, msm))}
        else:
            e2e = {"value": None, "unit": "MSM/s", "h2d_bytes_per_step": int(n_total * 128), "d2h_bytes_per_step": 144 * world,
                   "note": f"host-pointer e2e failed on a rank: {failed}"}
    elif world > 1:
        e2e = {"value": None, "unit": "MSM/s", "h2d_bytes_per_step": int(n * 128), "d2h_bytes_per_step": 144,
               "note": "--skip-e2e"}

    outputs = {"msm_bls12_381_affine": affine_words(result, P_BLS, 6)}

    # ---------------------------------------------------------------- Goldilocks NTT (second half of the metric)
    ntt_res = bench_ntt(args, torch, ntt, _lib, peak, peak_src, barrier, max_over_ranks, world, outputs)

    # ---------------------------------------------------------------- config 4: Pallas MSM, sharded like the headline
    pallas = bench_pallas(args, torch, msm, parallel, barrier, max_over_ranks, rank, world, outputs)

    # ---------------------------------------------------------------- the reference's own sm_100a kernels (N = 1)
    ref_gpu = None
    if world == 1 and need_host and not args.skip_ref_gpu:
        ref_gpu = bench_reference_gpu(args, torch, msm, ntt, _lib, pts_host, sc_host, e2e_result, e2e)

    # ---------------------------------------------------------------- CPU baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        lg_s = min(args.lg_cpu_sample, args.lg_msm)
        ns = 1 << lg_s
        cores = os.cpu_count() or 1
        hp = pts_host[:ns] if need_host else np.tile(base, (ns // m, 1))
        _, dt, kind = cpu_reference_msm(np.ascontiguousarray(hp), np.ascontiguousarray(sc_host[:ns]), cores)
        cpu = {"value": (ns / dt) / n_total, "unit": "MSM/s", "cores": cores, "kind": kind,
               "sample": f"one 2^{lg_s}-point MSM ({dt:.2f} s) on {cores} host threads, scaled by point "
                         f"throughput to 2^{args.lg_msm}; sppark msm/pippenger.hpp on portable (non-blst) arithmetic"}

    if rank == 0:
        line = {"metric": f"BLS12-381 G1 MSM/s @2^{args.lg_msm} points", "value": value, "unit": "MSM/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u32x12 (384-bit Montgomery integers)", "data": "synthetic",
                "config": {"workload": f"bls12_381_g1_msm_2^{args.lg_msm}",
                           "points": f"(i+1)*G, 2^{min(LG_DISTINCT, args.lg_msm)} distinct, replicated",
                           "scalars": "uniform < 2^254, seed 42+rank", "sharding": f"point-chunk x{world}, all-gather of partials",
                           "l2": "inputs (8.6 GB at 2^26) exceed L2; no flush needed"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches), "roofline": roofline,
                "cpu_baseline": cpu, "check": check, "ntt": ntt_res, "pallas_msm": pallas,
                "reference_gpu": ref_gpu}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def phases_entries(n, world):
    """mixed additions of one accumulate launch: one per (point, window), c chosen as the library does."""
    best = None
    for c in range(4, 23):
        w = (256 + c - 1) // c
        cost = w * (1.11 * n + 5.5 * (1 << (c - 1)))
        if best is None or cost < best[0]:
            best = (cost, w)
    return best[1] * n


def _jac_equal(a, b, msm, field=0, nl=6):
    """Equality of two Jacobian points as group elements, by cross-multiplied coordinates
    (X1*Z2^2 == X2*Z1^2, Y1*Z2^3 == Y2*Z1^3), using the library's own field multiply (no oracle
    on this path).  field / nl: selftest field id and 64-bit limbs per coordinate (0 / 6 =
    BLS12-381 fp, 2 / 4 = Pallas fp)."""
    a = np.asarray(a, dtype=np.uint64)
    b = np.asarray(b, dtype=np.uint64)
    za, zb = a[2 * nl:], b[2 * nl:]
    if not za.any() or not zb.any():
        return (not za.any()) and (not zb.any())
    mul = lambda x, y: msm.selftest_field(field, "mul", x.reshape(1, nl), y.reshape(1, nl))[0]   # noqa: E731
    za2, zb2 = mul(za, za), mul(zb, zb)
    if not np.array_equal(mul(a[:nl], zb2), mul(b[:nl], za2)):
        return False
    return np.array_equal(mul(a[nl:2 * nl], mul(zb2, zb)), mul(b[nl:2 * nl], mul(za2, za)))


P_BLS = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
P_PALLAS = 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001   # base field of Pallas
NTT_DUMP_SAMPLE = 1 << 20        # Goldilocks NTT positions written by --dump-outputs


def words32(a):
    """uint64 array (..., k) -> (..., 2k) float64 of its little-endian 32-bit words (exact)."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.view(np.uint32).reshape(*a.shape[:-1], 2 * a.shape[-1]).astype(np.float64)


def affine_words(jac, p, nl):
    """Jacobian point of the library (X, Y, Z Montgomery residues, nl 64-bit limbs each) -> the
    affine x = X/Z^2, y = Y/Z^3 as plain integers, (2, 2*nl) float64 32-bit words; the point at
    infinity is all zeros.  Unlike the Jacobian coordinates, which depend on the order the
    buckets were summed in, this is the same for every computation of the same group element."""
    jac = np.asarray(jac, dtype=np.uint64)
    rinv = pow(1 << (64 * nl), -1, p)
    X, Y, Z = (sum(int(v) << (64 * i) for i, v in enumerate(jac[k * nl:(k + 1) * nl])) * rinv % p for k in range(3))
    xy = [0, 0]
    if Z:
        zi = pow(Z, -1, p)
        xy = [X * zi * zi % p, Y * zi * zi * zi % p]
    limbs = np.array([[(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(nl)] for v in xy], dtype=np.uint64)
    return words32(limbs)


def dump_outputs(outdir, outputs):
    """--dump-outputs: every array of `outputs` as outdir/<name>.npy.  All values are float64
    holding integers below 2^53 exactly, so two builds can be compared array for array:
      msm_bls12_381_affine   the headline MSM's group element (affine_words)
      pallas_msm_affine      the Pallas MSM's group element
      ntt_goldilocks         Goldilocks NTT output, (k, 2) 32-bit words, at the positions in
      ntt_goldilocks_index   (all of them up to 2^20 points, else 2^20 drawn with seed 0)
    The NTT transforms its buffer in place, so its array is the seeded input transformed
    max(3, --warmup) + --steps times.  The NTT arrays are written by single-rank runs only: with
    several ranks each holds a slab of a sharded transform."""
    os.makedirs(outdir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(outdir, name + ".npy"), np.asarray(a, dtype=np.float64))


R_PALLAS = 0x40000000000000000000000000000000224698fc0994a8dd8c46eb2100000001   # order of the Pallas group


def bench_pallas(args, torch, msm, parallel, barrier, max_over_ranks, rank, world, outputs):
    """BASELINE.json config 4: Pallas MSM over 2^24 points, sharded by point-chunk over the ranks
    (2^21 points per GPU at N = 8), one all-gather of the 96-byte partial results + combine.
    Device-resident, strong scaling; checked by folding every rank's scalars onto the distinct
    points (same size-independent property as the headline)."""
    try:
        lg = args.lg_pallas
        n = (1 << lg) // world
        m = 1 << min(LG_DISTINCT, lg - (world.bit_length() - 1))
        base_dev = msm.generate_points_dev(msm.PALLAS, m)
        rng = np.random.default_rng(4242 + rank)
        sc = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
        sc[:, 3] >>= np.uint64(2)                                      # < 2^254 < group order
        d_points = base_dev.repeat(n // m, 1).contiguous()
        d_scalars = torch.from_numpy(sc.view(np.int64)).cuda()

        def step():
            return parallel.msm_sharded(lambda: msm.msm_dev(msm.PALLAS, d_points, d_scalars),
                                        lambda parts: msm.combine(msm.PALLAS, parts) if world > 1 else parts[0],
                                        12, device="cuda")
        for _ in range(max(3, args.warmup)):
            result = step()
        barrier()
        iters = args.steps
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            result = step()
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1) / iters)
        outputs["pallas_msm_affine"] = affine_words(result, P_PALLAS, 4)
        folded = fold_scalars(sc, m, R_PALLAS)
        if world > 1:
            parts = parallel.all_gather_partials(folded.reshape(-1), "cuda").reshape(world * m, 4)
            folded = fold_scalars(np.ascontiguousarray(parts), m, R_PALLAS)
        small = msm.msm_dev(msm.PALLAS, base_dev, torch.from_numpy(folded.view(np.int64)).cuda())
        ok = _jac_equal(result, small, msm, field=2, nl=4)
        del d_points, d_scalars
        torch.cuda.empty_cache()
        return {"metric": f"Pallas MSM/s @2^{lg} points", "value": 1e3 / ms, "unit": "MSM/s", "ms_per_step": ms,
                "scaling": "strong", "n_gpus": world, "points_per_gpu": n,
                "sharding": f"point-chunk x{world}, all-gather of 96-byte partials + combine",
                "check": f"folded-msm over {world} rank(s) " + ("ok" if ok else "MISMATCH")}
    except Exception as e:                                             # never take the headline down
        return {"metric": "Pallas MSM/s", "value": None, "error": f"{type(e).__name__}: {e}"}


class _RustError(C.Structure):
    _fields_ = [("code", C.c_int), ("message", C.c_void_p)]


def bench_reference_gpu(args, torch, msm, ntt, _lib, pts_host, sc_host, ours_result, ours_e2e):
    """The kernels to beat: the REFERENCE's own CUDA code (poc/msm-cuda/cuda/pippenger.cu and
    poc/ntt-cuda/cuda/ntt_api.cu) compiled for sm_100a into oracle/_ref by oracle/Makefile, called
    through the identical host-pointer entry points on the same buffers, pinned and pageable, and
    (NTT) on device-resident data.  Runs after the repository's own timed regions; rank 0, N = 1."""
    out = {"source": "oracle/_ref/*.so = the reference's sources built with nvcc -arch sm_100a (oracle/Makefile)"}
    refdir = os.path.join(ROOT, "oracle", "_ref")
    n = pts_host.shape[0]
    try:
        path = os.path.join(refdir, "libref_msm_gpu.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        ref = C.CDLL(path)
        ref.mult_pippenger.restype = _RustError
        ref.mult_pippenger.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]

        def ref_msm(p, s_):
            o_ = np.zeros(18, dtype=np.uint64)
            e = ref.mult_pippenger(o_.ctypes.data, p.ctypes.data, n, s_.ctypes.data)
            if e.code != 0:
                raise RuntimeError(f"reference mult_pippenger returned {e.code}")
            return o_

        def clock(fn, reps):
            fn()
            t0 = time.perf_counter()
            for _ in range(reps):
                r_ = fn()
            return (time.perf_counter() - t0) / reps, r_

        reps = args.steps
        dt_ref_pin, r_ref = clock(lambda: ref_msm(pts_host, sc_host), reps)
        pts_pg, sc_pg = np.array(pts_host), np.array(sc_host)            # pageable copies (a Rust Vec is pageable)
        dt_ref_pg, _ = clock(lambda: ref_msm(pts_pg, sc_pg), reps)
        dt_our_pg, r_our = clock(lambda: msm.multi_scalar_mult(pts_pg, sc_pg), reps)
        del pts_pg, sc_pg
        out["msm"] = {"workload": f"bls12_381_g1_msm_2^{args.lg_msm}, mult_pippenger(host pointers)",
                      "reference_ms": {"pinned": dt_ref_pin * 1e3, "pageable": dt_ref_pg * 1e3},
                      "ours_ms": {"pinned": ours_e2e["ms_per_step"], "pageable": dt_our_pg * 1e3},
                      "speedup": {"pinned": dt_ref_pin * 1e3 / ours_e2e["ms_per_step"], "pageable": dt_ref_pg / dt_our_pg},
                      "same_group_element": bool(_jac_equal(r_ref, ours_result, msm) and _jac_equal(r_our, r_ref, msm))}
    except Exception as e:
        out["msm"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        path = os.path.join(refdir, "libref_ntt_gl64_gpu.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        ref = C.CDLL(path)
        ref.ref_ntt_stream.restype = C.c_void_p
        ref.ref_ntt_dev_async.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]
        ref.compute_ntt.restype = _RustError
        ref.compute_ntt.argtypes = [C.c_size_t, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]
        rs = torch.cuda.ExternalStream(ref.ref_ntt_stream())
        cur = torch.cuda.current_stream()
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        l = _lib.lib()
        res = {}
        for lg in sorted({20, args.lg_ntt}):
            nn = 1 << lg
            rng = np.random.default_rng(70 + lg)
            host = rng.integers(0, GL_P, size=nn, dtype=np.uint64)
            row = {}
            for order, name in ((0, "NN"), (1, "NR"), (2, "RN")):
                d1 = torch.from_numpy(host.view(np.int64)).cuda()
                d2 = d1.clone()
                p1, p2 = d1.data_ptr(), d2.data_ptr()

                def timed(fn, stream, iters=args.steps):
                    for _ in range(3):
                        fn()
                    torch.cuda.synchronize()
                    tot = 0.0
                    for _ in range(iters):
                        flush.zero_()
                        torch.cuda.synchronize()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(stream)
                        fn()
                        e1.record(stream)
                        e1.synchronize()
                        tot += e0.elapsed_time(e1)
                    return tot / iters * 1e3
                ours_us = timed(lambda: l.sppark_b200_ntt_dev(0, p1, lg, order, 0, 0, cur.cuda_stream), cur)
                ref_us = timed(lambda: ref.ref_ntt_dev_async(p2, lg, order, 0, 0), rs)
                d1.copy_(torch.from_numpy(host.view(np.int64)))
                d2.copy_(d1)
                torch.cuda.synchronize()
                l.sppark_b200_ntt_dev(0, p1, lg, order, 0, 0, cur.cuda_stream)
                ref.ref_ntt_dev_async(p2, lg, order, 0, 0)
                torch.cuda.synchronize()
                row[name] = {"ours_us": ours_us, "reference_us": ref_us, "speedup": ref_us / ours_us,
                             "bit_identical": bool(torch.equal(d1, d2))}
            res[f"lg{lg}_device_resident"] = row
        # host-pointer compute_ntt at the metric size: pinned and pageable
        nn = 1 << args.lg_ntt
        pin_t = torch.empty(nn, dtype=torch.int64, pin_memory=True)
        pin = pin_t.numpy().view(np.uint64)
        pin[:] = np.random.default_rng(9).integers(0, GL_P, size=nn, dtype=np.uint64)
        pg = np.array(pin)

        def host_ms(fn, buf, reps=args.steps):
            fn(buf)
            t0 = time.perf_counter()
            for _ in range(reps):
                fn(buf)
            return (time.perf_counter() - t0) / reps * 1e3

        def ref_host(buf):
            e = ref.compute_ntt(0, buf.ctypes.data, args.lg_ntt, 0, 0, 0)
            assert e.code == 0
        res[f"lg{args.lg_ntt}_compute_ntt_host_ms"] = {
            "ours": {"pinned": host_ms(lambda b: ntt.NTT(0, b, ntt.NN), pin), "pageable": host_ms(lambda b: ntt.NTT(0, b, ntt.NN), pg)},
            "reference": {"pinned": host_ms(ref_host, pin), "pageable": host_ms(ref_host, pg)}}
        out["ntt"] = res
    except Exception as e:
        out["ntt"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        out["polynomial"] = bench_polynomial(args, torch, _lib, refdir)
    except Exception as e:
        out["polynomial"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def bench_polynomial(args, torch, _lib, refdir):
    """SURVEY.md section 8 row f4 next to the reference's own polynomial/ kernels (oracle/ref_poly.cu
    built for sm_100a): Goldilocks, 2^lg_ntt elements resident in HBM (128 MiB at 2^24, larger
    than L2), CUDA events on the stream each side launches on, mean of --steps calls back to back."""
    path = os.path.join(refdir, "libref_poly_gl64_gpu.so")
    if not os.path.exists(path):
        raise FileNotFoundError(path)
    ref = C.CDLL(path)
    ref.ref_poly_stream.restype = C.c_void_p
    ref.ref_prefix_op_dev.argtypes = [C.c_int, C.c_void_p, C.c_size_t]
    ref.ref_div_by_x_minus_z_dev.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
    ref.ref_evaluate_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    l = _lib.lib()
    n = 1 << args.lg_ntt
    host = np.random.default_rng(11).integers(0, GL_P, size=n, dtype=np.uint64)
    d = torch.from_numpy(host.view(np.int64)).cuda()
    z = np.array([123456789], dtype=np.uint64)
    xs = torch.tensor([3], dtype=torch.int64, device="cuda")
    r1, r2 = torch.zeros_like(xs), torch.zeros_like(xs)
    cur, rs = torch.cuda.current_stream(), torch.cuda.ExternalStream(ref.ref_poly_stream())
    s = cur.cuda_stream

    def timed(fn, stream, iters=args.steps):
        for _ in range(3):
            fn()
        stream.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / iters * 1e3

    rows = {}
    for name, mine, theirs in (
            ("prefix_add", lambda: l.sppark_b200_prefix_op_dev(0, 0, d.data_ptr(), d.data_ptr(), n, s),
             lambda: ref.ref_prefix_op_dev(0, d.data_ptr(), n)),
            ("prefix_multiply", lambda: l.sppark_b200_prefix_op_dev(0, 1, d.data_ptr(), d.data_ptr(), n, s),
             lambda: ref.ref_prefix_op_dev(1, d.data_ptr(), n)),
            ("div_by_x_minus_z", lambda: l.sppark_b200_div_by_x_minus_z_dev(0, d.data_ptr(), n, z.ctypes.data, 0, s),
             lambda: ref.ref_div_by_x_minus_z_dev(d.data_ptr(), n, z.ctypes.data, 0)),
            ("evaluate_1_point", lambda: l.sppark_b200_evaluate_dev(0, r1.data_ptr(), xs.data_ptr(), 1, d.data_ptr(), n, s),
             lambda: ref.ref_evaluate_dev(r2.data_ptr(), xs.data_ptr(), 1, d.data_ptr(), n))):
        ours_us, ref_us = timed(mine, cur), timed(theirs, rs)
        rows[name] = {"ours_us": ours_us, "reference_us": ref_us, "speedup": ref_us / ours_us}
    torch.cuda.synchronize()
    rows["evaluate_1_point"]["same_value"] = bool(torch.equal(r1, r2))
    # the two sides' division of the same polynomial, bit for bit
    a = torch.from_numpy(host.view(np.int64)).cuda()
    b = a.clone()
    _lib.check(l.sppark_b200_div_by_x_minus_z_dev(0, a.data_ptr(), n, z.ctypes.data, 0, s))
    if ref.ref_div_by_x_minus_z_dev(b.data_ptr(), n, z.ctypes.data, 0) != 0:
        raise RuntimeError("reference div_by_x_minus_z failed")
    torch.cuda.synchronize()
    rows["div_by_x_minus_z"]["bit_identical"] = bool(torch.equal(a, b))
    return {"workload": f"Goldilocks, 2^{args.lg_ntt} elements, device resident", **rows}


def bench_ntt(args, torch, ntt, _lib, peak, peak_src, barrier, max_over_ranks, world, outputs):
    """Goldilocks 2^lg NTT, NN order, device-resident (NTT::Base_dev_ptr path) and e2e
    (compute_ntt with a pinned host buffer).  With N > 1 ranks ONE transform is slab-sharded over
    the ranks (column slabs, one NCCL all-to-all between the two local passes; strong scaling)."""
    lg = args.lg_ntt
    n = 1 << lg
    if world > 1:
        return bench_ntt_sharded(args, torch, _lib, peak, peak_src, barrier, max_over_ranks, world)
    rng = np.random.default_rng(7)
    host_t = torch.empty(n, dtype=torch.int64, pin_memory=True)
    host = host_t.numpy().view(np.uint64)
    host[:] = rng.integers(0, GL_P, size=n, dtype=np.uint64)
    d = host_t.cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    iters = args.steps
    for _ in range(max(3, args.warmup)):
        ntt.ntt_dev(d, ntt.NN)
    barrier()
    tot = 0.0
    for _ in range(iters):
        flush.zero_()                                                   # evict L2 between iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ntt.ntt_dev(d, ntt.NN)
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    ms = max_over_ranks(tot / iters)
    if args.dump_outputs:            # d holds the last timed transform's output until the profiled one below
        idx = np.arange(n) if n <= NTT_DUMP_SAMPLE else \
            np.sort(np.random.default_rng(0).choice(n, NTT_DUMP_SAMPLE, replace=False))
        outputs["ntt_goldilocks_index"] = idx
        outputs["ntt_goldilocks"] = words32(d[torch.from_numpy(idx).cuda()].cpu().numpy().view(np.uint64)[:, None])
    _lib.profile_enable(True)
    flush.zero_()
    ntt.ntt_dev(d, ntt.NN)
    torch.cuda.synchronize()
    passes = [v for _, v in _lib.profile_read()]
    _lib.profile_enable(False)
    alg = 2 * n * 8
    worst = max(passes) if passes else ms
    res = {"metric": f"Goldilocks NTT/s @2^{lg} (NN, forward)", "value": world * 1e3 / ms, "unit": "NTT/s",
           "ms_per_ntt": ms, "scaling": "replicas", "iters": iters, "l2": "256 MiB write between iterations",
           "roofline": {"bound": "hbm", "kernel": "ntt::pass_kernel_static<gl64, 12 x 2> (slowest of the two block-tile passes)",
                        "achieved": alg / (worst * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (worst * 1e-3) / 1e9 / peak,
                        # dram__bytes_read.sum + dram__bytes_write.sum of that pass from the ncu --set full
                        # capture (profiles/ntt_block_r02.md, launch 0: 134.4 MB + 87.6 MB), 2^24 only
                        "traffic": 222.1e6 if lg == 24 else None, "traffic_source": "profiles/ntt_block_r02.md",
                        "peak_source": peak_src,
                        # the binding resource is the INT32 ALU pipe, not HBM: the butterfly network alone
                        # (tools/gl64_bfly_bench.cu, profiles/gl64_butterfly_microbench_r02.txt) needs 37.9
                        # SMSP-cycles per butterfly at 90 % ALU-pipe utilisation
                        "int32_alu": {"butterflies": n // 2 * lg, "dense_cycles_per_butterfly": 37.9,
                                      "floor_ms": (n // 2 * lg / 32) * 37.9 / (148 * 4) / 1.965e6,
                                      "frac": ((n // 2 * lg / 32) * 37.9 / (148 * 4) / 1.965e6) / ms},
                        "pass_ms": [round(p, 4) for p in passes],
                        "whole_transform_frac": alg / (ms * 1e-3) / 1e9 / peak}}
    # e2e: in place on the pinned host buffer through compute_ntt
    ntt.NTT(0 if world == 1 else torch.cuda.current_device(), host, ntt.NN)
    t0 = time.perf_counter()
    reps = args.steps
    for _ in range(reps):
        ntt.NTT(0 if world == 1 else torch.cuda.current_device(), host, ntt.NN)
    dt = (time.perf_counter() - t0) / reps
    res["e2e"] = {"value": 1.0 / dt, "unit": "NTT/s", "h2d_bytes_per_step": n * 8, "d2h_bytes_per_step": n * 8,
                  "api": "compute_ntt (host pointer, pinned)"}
    return res


def bench_ntt_sharded(args, torch, _lib, peak, peak_src, barrier, max_over_ranks, world):
    """ONE transform slab-sharded over the ranks.  Headline: Goldilocks 2^lg.  Also reported
    (SURVEY.md section 8d config 5): BabyBear 2^27, the largest transform that field admits
    (p - 1 = 15 * 2^27; "2^28" is not a valid BabyBear domain), 2^9 x 2^18 with a two-pass second
    stage."""
    import torch.distributed as dist
    from sppark_b200 import parallel
    rank = dist.get_rank()
    lg_g = world.bit_length() - 1
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(step, iters):
        for _ in range(max(3, args.warmup)):
            step()
        barrier()
        tot = 0.0
        for _ in range(iters):
            flush.zero_()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            e1.synchronize()
            tot += max_over_ranks(e0.elapsed_time(e1))
        return tot / iters

    def run(fid, lg, name, esz, iters):
        n_local = (1 << lg) // world
        rng = np.random.default_rng(7 + rank)
        if fid == 0:
            local = torch.from_numpy(rng.integers(0, GL_P, size=n_local, dtype=np.uint64).view(np.int64)).cuda()
        else:
            local = torch.from_numpy(rng.integers(0, 0x78000001, size=n_local, dtype=np.uint32).view(np.int32)).cuda()
        pass_fn = parallel.gpu_slab_pass(fid, lg, lg_g, rank)
        # baseline exchange: staging buffer + NCCL all-to-all between the two local stages
        ms_nccl = timed(lambda: parallel.ntt_slab(local, lg, fid, pass_fn), iters)
        # fused exchange: stage 1 stores straight into the receivers over NVLink peer memory
        exchange, ms, why = "NCCL all_to_all_single", ms_nccl, None
        if os.environ.get("SPPARK_B200_NTT_EXCHANGE", "p2p") == "p2p":
            ok = torch.ones(1, dtype=torch.int32, device="cuda")
            peers = None
            try:
                peers = parallel.SlabPeers(n_local * esz)
                scratch = torch.empty_like(local)
                ref = parallel.ntt_slab(local, lg, fid, pass_fn)
                got = parallel.ntt_slab_p2p(local, lg, fid, rank, peers, scratch)
                if not torch.equal(ref, got):
                    raise RuntimeError("fused exchange result differs from the all-to-all route")
            except Exception as e:                       # e.g. no peer access between these GPUs
                why = f"{type(e).__name__}: {e}"
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)    # all ranks take the same route
            if int(ok.item()):
                ms = timed(lambda: parallel.ntt_slab_p2p(local, lg, fid, rank, peers, scratch), iters)
                exchange = "fused into stage 1: NVLink peer stores (CUDA IPC), 4-byte all-reduce as the barrier"
            if peers is not None:
                try:
                    peers.close()
                except Exception:
                    pass
        alg = 2 * (1 << lg) * esz
        n1 = 1 << parallel.slab_first_digit(lg, fid)
        return {"metric": f"{name} NTT/s @2^{lg} (NN, forward)", "value": 1e3 / ms, "unit": "NTT/s",
                "ms_per_ntt": ms, "scaling": "strong", "iters": iters,
                "sharding": f"column slabs x{world} of a {n1} x {(1 << lg) // n1} matrix, "
                            f"{n_local * esz * (world - 1) // world} B per rank cross NVLink",
                "exchange": exchange, "ms_with_nccl_all_to_all": ms_nccl, "fused_exchange_error": why,
                "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak * world, "unit": "GB/s",
                             "frac": alg / (ms * 1e-3) / 1e9 / (peak * world), "traffic": None, "peak_source": peak_src},
                "e2e": None}

    res = run(0, args.lg_ntt, "Goldilocks", 8, args.steps)
    res["babybear_2pow27"] = run(1, 27, "BabyBear", 4, args.steps)
    return res


if __name__ == "__main__":
    main()
