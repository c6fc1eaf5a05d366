#!/usr/bin/env python
"""bench.py — ICP + covariance scan pairs/s of the scan-matching path (BASELINE.json metric).

A "step" is one pass of the hot path (DpgSLAM::runIcp + calculate_ICP_COV semantics, reference
src/dpg_slam/dpg_slam.cc:362-446) over one batch of synthetic Hokuyo-like scan pairs.

  workloads  corridor      BASELINE configs[1]: 5000 sequential odometry pairs per GPU (weak scaling)   <- headline
             loop_closure  BASELINE configs[2]: 100k loop-closure candidates per GPU (weak); at N = 1 the default
                           run measures it too and reports it under "also"
             dense         BASELINE configs[3]: 4096-beam scans, point-to-line, ONE global batch of 1M pairs sharded
                           over the GPUs (strong scaling)
             multisession  BASELINE configs[4]: 8 sessions x 50k scans on a shared, partly changed world; the
                           candidate list of one reoptimize() (gates 5 m / 2 m) is enumerated ON the devices and
                           sharded round-robin (strong scaling); the pair count is reported
  settings   1081 (4096) beams, every point enters ICP (downsample divisor 1), reciprocal correspondences,
             covariance = the intended Censi form on the final ICP correspondences (CENSI_CORR), all other
             parameters the reference's defaults (500 iterations max, 0.6 m gate, eps 5e-9).
  value      pairs/s with the scan store and pair list already resident in HBM; CUDA events on the launching
             stream, L2 flushed between steps, max over ranks.
  e2e        the same batch through the public API with HOST buffers every step: raw ranges H2D + on-device
             scan->cloud + pair list H2D (or node table H2D + on-device enumeration) + ICP/covariance + records D2H;
             at N > 1 it includes the cross-rank synchronisation and rank 0's copy of the WHOLE gathered batch.
  N > 1      pairs sharded round-robin (pair k -> rank k % N), scan store replicated, records gathered by peer stores
             from the kernel epilogue (no collective on the data path; DPGICP_BENCH_GATHER=nccl for the all-gather).
  checks     in the run: records of the e2e arm == resident arm; the gathered buffer holds every rank's records;
             rank 0 re-aligns a strided sample of the GLOBAL batch on its one GPU and compares with the gathered
             records bit for bit (1 GPU == N GPUs); a strided sample equals the CPU oracle bit for bit.
  outputs    --dump-outputs DIR (one GPU): the records of the last timed step, one DIR/<field>.npy per record field plus
             index.npy (their positions in the batch); inputs are seeded, so two builds can be compared output for output.

`--impl reference` times the reference's CPU algorithm on the host cores (the oracle port, oracle/dpg_oracle.c,
OpenMP over pairs): PCL itself cannot be built in this image (DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "icp_cov_scan_pairs_per_sec"
UNIT = "pairs/s"
WORKLOADS = {
    "corridor": dict(desc="BASELINE configs[1]: synthetic corridor trajectory, 5000 sequential odometry scan pairs per GPU",
                     scaling="weak", pairs_per_gpu=5000, beams=1081, seed=2, metric=0),
    "loop_closure": dict(desc="BASELINE configs[2]: loop-closure candidate sweep, 100k scan pairs over 2000 scans with random "
                              "initial offsets, per GPU", scaling="weak", pairs_per_gpu=100_000, n_scans=2000, beams=1081, seed=3, metric=0),
    "dense": dict(desc="BASELINE configs[3]: dense 4096-beam scans, point-to-line, 1M pairs over 20000 scans, ONE global batch "
                       "sharded over the GPUs", scaling="strong", global_pairs=1_000_000, n_scans=20_000, beams=4096, seed=4, metric=1),
    "multisession": dict(desc="BASELINE configs[4]: dynamic-environment multi-session map, 8 sessions x 50k scans, gated all-pairs "
                              "candidates (5 m same session / 2 m across) of one reoptimize(), enumerated on the devices",
                         scaling="strong", sessions=8, scans_per_session=50_000, beams=1081, seed=5, metric=0),
}
FLUSH_BYTES = 512 << 20


# ---- workload ----------------------------------------------------------------------------------------------
def make_host_workload(name: str, n_pairs: int, rank=0, world=1):
    """corridor / loop_closure / dense: host pair list + raw ranges (replicated on every rank)."""
    from dpg_slam_b200 import synth
    w = WORKLOADS[name]
    if name == "corridor":
        return synth.config_corridor(n_pairs=n_pairs, n_beams=w["beams"], seed=w["seed"])
    return synth.config_loop_closure(n_pairs=n_pairs, n_scans=w["n_scans"], n_beams=w["beams"], seed=w["seed"])


def bench_params(name: str, search: str):
    from dpg_slam_b200._abi import COV_CENSI_CORR, SEARCH_PROJECTIVE, SEARCH_PRUNED, Params
    return Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR, metric=WORKLOADS[name]["metric"],
                           search=SEARCH_PROJECTIVE if search == "projective" else SEARCH_PRUNED)


def gather_desc(world: int) -> str:
    if world == 1:
        return "none (1 GPU)"
    return ("NCCL all_gather" if os.environ.get("DPGICP_BENCH_GATHER", "fused") == "nccl"
            else "peer stores from the kernel epilogue (fused)")


def workload_config(name: str, n_gpus: int, global_pairs: int, search: str, extra=None):
    w = WORKLOADS[name]
    cfg = {"workload": w["desc"], "global_pairs": int(global_pairs),
           "pairs_per_gpu": int(global_pairs // n_gpus), "beams": w["beams"],
           "fov_deg": 270, "downsample_divisor": 1, "metric_kind": "point_to_line" if w["metric"] else "point_to_point",
           "reciprocal": True, "cov_mode": "CENSI_CORR(cap 200)", "max_iterations": 500, "max_correspondence_distance_m": 0.6,
           "search": ("exact pruned (bounding-box groups)" if search == "pruned" else
                      "PROJECTIVE (approximate: beam-order projection, window 8 each side; not the reference's exact search)"),
           "sharding": f"round-robin over {n_gpus} GPU(s), scan store replicated",
           "l2": "flushed between timed steps (512 MiB memset outside the event pair)", "seed": w["seed"],
           "gather": gather_desc(n_gpus)}
    if extra:
        cfg.update(extra)
    return cfg


# ---- clocks --------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU baseline / reference arm ---------------------------------------------------------------------------
def host_threads() -> int:
    """all host cores, whatever OMP_NUM_THREADS says (torch.distributed.run sets it to 1)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def cpu_sample_run(src, tgt, guess, pts, off, p, idx, threads):
    from oracle import oracle_py as O
    t0 = time.perf_counter()
    rec, used = O.run_batch(pts, off, src[idx], tgt[idx], guess[idx], p, fast=1, threads=threads)
    return time.perf_counter() - t0, used, rec


def choose_cpu_sample(src, tgt, guess, pts, off, p, threads, target_s=12.0):
    """Bounded sample of the workload: pilot on 4 pairs per core, then size for ~target_s of CPU time."""
    n = len(src)
    pilot = np.linspace(0, n - 1, min(n, 4 * threads)).astype(np.int64)
    dt, _, _ = cpu_sample_run(src, tgt, guess, pts, off, p, pilot, threads)
    per_pair = dt / len(pilot)
    m = int(max(len(pilot), min(n, target_s / max(per_pair, 1e-9))))
    return np.linspace(0, n - 1, m).astype(np.int64)


def oracle_clouds(ranges, scanner):
    from oracle import oracle_py as O
    return O.clouds_from_ranges(ranges, scanner)


def reference_workload(args):
    """(src, tgt, guess, ranges, scanner, global_pairs) for the reference arm: the product arm's workload, with the big
    strong-scaling configs cut down to what the bounded CPU sample needs."""
    from dpg_slam_b200 import synth
    w = WORKLOADS[args.workload]
    world = args.gpus
    if args.workload in ("corridor", "loop_closure"):
        n_global = (args.pairs or w["pairs_per_gpu"]) * world
        wl = make_host_workload(args.workload, n_global)
        return wl.src_idx, wl.tgt_idx, wl.guess, wl.ranges, wl.scanner, n_global, "evenly strided"
    if args.workload == "dense":
        n_global = args.pairs or w["global_pairs"]
        # the CPU can only afford a few hundred 4096-beam pairs: the same generator at 1/50 of the scans and pairs
        wl = synth.config_loop_closure(n_pairs=max(2000, n_global // 50), n_scans=max(200, w["n_scans"] // 50), n_beams=w["beams"], seed=w["seed"])
        return wl.src_idx, wl.tgt_idx, wl.guess, wl.ranges, wl.scanner, n_global, "same generator at 1/50 of the scans and pairs, evenly strided"
    sps = max(200, (args.scans_per_session or w["scans_per_session"]) // 50)
    wl = synth.config_multisession(n_sessions=w["sessions"], scans_per_session=sps, n_beams=w["beams"], seed=w["seed"],
                                   size=100.0 / np.sqrt(50.0), n_boxes=max(6, 300 // 50))
    from oracle import oracle_py as O
    src, tgt = O.enumerate_pairs(wl.poses_est[:, :2], wl.passes, 5.0, 2.0)
    wl = synth.with_pairs(wl, src, tgt)
    return wl.src_idx, wl.tgt_idx, wl.guess, wl.ranges, wl.scanner, len(src), \
        "same generator at 1/50 of the scans on 1/50 of the area (same node density), evenly strided"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import __graft_entry__ as g
    if not os.path.exists(os.path.join(ROOT, "oracle", "libdpgoracle.so")):
        g.build()
    src, tgt, guess, ranges, scanner, n_global, how = reference_workload(args)
    p = bench_params(args.workload, args.search)
    pts, off = oracle_clouds(ranges, scanner)
    threads = host_threads()
    idx = choose_cpu_sample(src, tgt, guess, pts, off, p, threads, target_s=float(os.environ.get("DPGICP_BENCH_CPU_TARGET_S", "8.0")))
    for _ in range(max(args.warmup, 0)):
        cpu_sample_run(src, tgt, guess, pts, off, p, idx[:max(8, len(idx) // 8)], threads)
    t_total, used = 0.0, threads
    for _ in range(args.steps):
        dt, used, _ = cpu_sample_run(src, tgt, guess, pts, off, p, idx, threads)
        t_total += dt
    value = len(idx) * args.steps / t_total
    sidx = idx[::max(1, len(idx) // 32)][:32]              # the reference itself is single-threaded (ros::spin)
    dt1, _, _ = cpu_sample_run(src, tgt, guess, pts, off, p, sidx, 1)
    sample = (f"{len(idx)} of the workload's pairs per step ({how}), oracle port with exact uniform-grid NN, "
              f"OpenMP over pairs on {used} threads (set explicitly: all host cores)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True,
            "scaling": WORKLOADS[args.workload]["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, args.gpus, n_global, args.search)
            if args.workload != "multisession" else multisession_config(args, args.gpus, None, args.search),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port", "sample": sample,
                             "single_thread_value": len(sidx) / dt1, "single_thread_sample": f"{len(sidx)} pairs, {dt1:.1f} s"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference = CPU restatement of runIcp + calculate_ICP_COV (PCL ICP is un-vendored and cannot be built here)"}
    print(json.dumps(line), flush=True)
    return 0


# ---- product arm: shared pieces ------------------------------------------------------------------------------------
def algorithmic_flops(rec, counts_s, counts_t, sum_corr):
    """SURVEY.md §8d normative work: I*(5*Ns*Nt + 8*Ns) + 14*sum K  +  60*N_H + 45*min(K,200)."""
    it = rec["iterations"].astype(np.float64)
    ns, nt = counts_s.astype(np.float64), counts_t.astype(np.float64)
    k_last = rec["n_correspondences"].astype(np.float64)
    icp = float(np.sum(it * (5.0 * ns * nt + 8.0 * ns)) + 14.0 * sum_corr)
    cov = float(np.sum(60.0 * k_last + 45.0 * np.minimum(k_last, 200.0)))
    return icp, cov


DUMP_BUDGET_BYTES = 60_000_000         # under 64 MB with the .npy headers
DUMP_FIELDS = (("tx", np.float32), ("ty", np.float32), ("theta", np.float32), ("rot_c", np.float32), ("rot_s", np.float32),
               ("iterations", np.float64), ("status", np.float64), ("n_correspondences", np.float64),    # integers, exact in f64
               ("mse", np.float64), ("cov", np.float64))
DUMP_RECORD_BYTES = 8 + sum(np.dtype(t).itemsize * (9 if f == "cov" else 1) for f, t in DUMP_FIELDS)     # + the index


def dump_sample(n_records: int) -> np.ndarray:
    """Sorted indices of the records --dump-outputs writes: all of them when they fit the budget, else a fixed seeded
    sample (the same for every run with the same arguments)."""
    k = DUMP_BUDGET_BYTES // DUMP_RECORD_BYTES
    if n_records <= k:
        return np.arange(n_records, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(n_records, size=k, replace=False)).astype(np.int64)


def dump_records(out_dir: str, rec, index) -> None:
    """The records a caller of the timed path receives, one float32/float64 array per field: <out_dir>/<field>.npy, plus
    index.npy, the position of each dumped record in the batch."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "index.npy"), np.asarray(index, np.float64))
    for f, t in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f"{f}.npy"), np.ascontiguousarray(rec[f], dtype=t))


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def fp32_peak(probe, nominal):
    """Rate of separately rounded binary32 multiplies and adds on this GPU, measured in this run: the scalar FMUL+FADD
    chains and the packed FMUL2 + packed-sum chains give the same ~37 T op/s (a packed instruction carries two results but
    takes two pipe cycles; it saves issue slots, not FP32 time).  Until round 2 the packed probe reported twice that:
    ptxas had contracted its mul.rn.f32x2 / add.rn.f32x2 pairs into single fused FFMA2 instructions."""
    measured = probe["mul_add_ops_per_s"] / 1e12
    packed = probe.get("mul_add_packed_ops_per_s", 0.0) / 1e12
    peak = max(measured, packed)
    return (peak if peak > 0 else nominal), measured, packed


def smem_block(counters, k_ms, sm_mhz, n_sm=148):
    """The other ceiling of the scan loop: every distance evaluation needs the searched point in the lane's registers —
    8 bytes per lane, 256 bytes per warp and point — and the shared-memory pipe writes back 128 bytes per cycle and SM
    (an LDS.128 occupies it for 4 cycles whether or not the address is a broadcast; ncu: lsu_writeback_active, profiles/).
    cycles = 2 per warp-level point evaluation."""
    warp_points = counters["distance_evals"] / 32.0
    cycles = 2.0 * warp_points
    avail = k_ms * 1e-3 * sm_mhz * 1e6 * n_sm
    return {"bound": "shared-memory write-back (LDS.128 broadcast of the searched points)", "cycles_per_warp_point": 2.0,
            "busy_cycles_per_launch": cycles, "available_cycles": avail, "frac": cycles / avail,
            "note": "distance loop only; box tests, seeds and moments add a few percent (ncu l1tex__lsu_writeback_active)"}


def roofline_block(name, search, k_ms, stage_ms, counters, rec_local, ns, nt, probe, peaks):
    """FP32 roofline of icp_pairs_kernel for rank 0's launch.  `achieved` is the EXECUTED FP32 work (the distance
    arithmetic the kernel really issued, counted on the device) over the live kernel time, against the measured rate of
    the instruction mix the bit-exact loop may use (separately rounded multiplies and adds, no FMA): a fraction <= 1.  The
    exact pruned search skips most of the brute-force evaluations SURVEY 8d's normative formula counts; that ratio is
    reported as algorithmic_speedup, not folded into the fraction."""
    icp_fl, cov_fl = algorithmic_flops(rec_local, ns, nt, counters["correspondences"])
    alg_tflops = (icp_fl + cov_fl) / (k_ms * 1e-3) / 1e12
    exec_flops = 5.0 * counters["distance_evals"] + 9.0 * counters["box_tests"]
    exec_tflops = exec_flops / (k_ms * 1e-3) / 1e12
    sm_mhz = float(peaks.get("sm_max_mhz", 1965.0))
    nominal = 148 * 128 * sm_mhz * 1e6 / 1e12
    peak, measured, packed = fp32_peak(probe, nominal)
    alg_bytes = float(np.sum(8.0 * (ns + nt) + 20 + 112))
    traffic, traffic_source, ncu_inst = None, None, None
    prof_name = {"corridor": "r02_final_icp_kernel_ncu.json"}.get(name)
    if prof_name and search == "pruned":
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", prof_name)))
            traffic = prof.get("dram_bytes_per_launch")
            ncu_inst = prof.get("instructions_executed")
            traffic_source = f"static: profiles/{prof_name} (ncu --set full capture of this workload's step, not measured in this run)"
        except Exception:
            pass
    out = {"kernel": "dpg::icp_pairs_kernel<WARPS,SEARCH,CLUSTER> (persistent CTAs; one step = a chain of up to 4 launches with growing "
                     "warps per pair, the last as 4-CTA clusters, timed together)",
           "bound": "fp32", "achieved": exec_tflops, "peak": peak, "unit": "TFLOP/s", "frac": exec_tflops / peak,
           "achieved_definition": "EXECUTED FP32 work: (5 flop x distance evaluations + 9 flop x box lower bounds) counted on the device "
                                  "/ live kernel time (CUDA events on the launching stream)",
           "peak_source": "measured on this GPU in this run (dpgicp_fp32_probe / dpgicp_fp32x2_probe): separately rounded multiply+add "
                          "chains, scalar and packed alike (the bit-exact distance loop may not use FMA; a packed instruction carries two "
                          "results but takes two pipe cycles); MEASURED_PEAKS.json has no FP32 figure; nominal rate 148 SM x 128 lanes x "
                          f"{sm_mhz} MHz = {nominal:.1f}",
           "algorithmic_tflops": alg_tflops, "algorithmic_speedup": (icp_fl + cov_fl) / max(exec_flops, 1.0),
           "algorithmic_definition": "SURVEY 8d brute-force flops I*(5*Ns*Nt+8*Ns)+14*K + 60*N_H+45*min(K,200) per kernel time; the exact "
                                     "pruned search executes 1/algorithmic_speedup of them",
           "kernel_ms": k_ms, "stage_ms": stage_ms, "traffic": traffic, "traffic_source": traffic_source,
           "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / (k_ms * 1e-3) / 1e9,
                   "peak_gbs": peaks.get("hbm_gbs"),
                   "frac": (alg_bytes / (k_ms * 1e-3) / 1e9) / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None},
           "fp32_probe_tops": {"mul_add": measured, "mul_add_packed": packed, "fma": probe["fma_ops_per_s"] / 1e12},
           "smem": smem_block(counters, k_ms, sm_mhz)}
    if ncu_inst:
        issue_peak = 4.0 * 148 * sm_mhz * 1e6
        out["issue_frac"] = ncu_inst / (k_ms * 1e-3) / issue_peak
        out["issue"] = {"warp_instructions_per_step": ncu_inst, "source": traffic_source, "peak_ginst_s": issue_peak / 1e9}
    return out


class Ctx:
    """per-process plumbing shared by the workloads"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.Stream(device=self.dev)
        self.flush = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, v: float) -> float:
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_values(self, vals):
        """every rank's list of floats, on every rank: [[rank 0's], [rank 1's], ...]"""
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [t.cpu().tolist()]
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [o.cpu().tolist() for o in out]

    def timed_steps(self, fn, steps):
        """`steps` calls of fn, each bracketed by CUDA events on the launching stream, L2 flushed before each (outside
        the event pair); returns (sum of device ms on this rank, wall seconds)"""
        torch = self.torch
        evs = []
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.flush.fill_(0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            fn()
            e1.record(self.stream)
            evs.append((e0, e1))
        self.barrier()
        return sum(a.elapsed_time(b) for a, b in evs), time.perf_counter() - t0

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def measure_host_list(cx: Ctx, sm, name, search, wl, n_global, steps, warmup, with_e2e=True, sampler=None):
    """Resident arm (+ e2e arm) of a host-pair-list workload on this process group.  Returns a dict of measurements
    (rank 0's view where per-rank) and the local records."""
    from dpg_slam_b200 import sharded
    torch = cx.torch
    p = bench_params(name, search)
    world, rank = cx.world, cx.rank
    shard = sharded.ShardedScanMatcher(sm, rank, world, None, cx.dev)
    idx = sharded.shard_indices(n_global, rank, world)
    n_beams = wl.ranges.shape[1]

    sm.upload_ranges(wl.ranges, wl.scanner)
    shard.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
    fused = world > 1 and os.environ.get("DPGICP_BENCH_GATHER", "fused") != "nccl"
    if fused:
        fused = shard.attach_fused_gather(n_global)           # False on every rank if a peer buffer could not be mapped

    def step_resident():
        shard.run(p)
        if world > 1 and not fused:
            shard.gather_device()

    # a step of the big strong-scaling batches takes seconds: their warm-up steps run on a prefix of every shard
    big = len(idx) * (n_beams / 1081.0) ** 2 > 150_000
    n_warm = min(len(idx), 20_000) if big else len(idx)
    for _ in range(max(warmup, 3)):
        if big:
            sm.run_range(p, 0, n_warm)
        else:
            step_resident()
    cx.barrier()
    launches0 = sm.last_run_counters()["kernel_launches"]
    dev_ms, t_wall = cx.timed_steps(step_resident, steps)
    launches = sm.last_run_counters()["kernel_launches"] - launches0
    counters = sm.last_run_counters()
    rec_local = sm.fetch_results()
    dev_ms_max = cx.max_over_ranks(dev_ms)
    value = n_global * steps / (dev_ms_max * 1e-3)

    # kernel-only duration (no gather) with per-stage events, for the roofline of the dominant kernel
    sm.enable_stage_timing(True)
    k_steps = 1 if big else max(3, min(steps, 10))
    k_list, stage_acc = [], None
    for _ in range(k_steps):
        cx.flush.fill_(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cx.stream); shard.run(p); e1.record(cx.stream)
        torch.cuda.synchronize(cx.dev)
        k_list.append(e0.elapsed_time(e1))
        st = sm.last_run_stage_ms()
        stage_acc = st if stage_acc is None else [a + b for a, b in zip(stage_acc, st)]
    sm.enable_stage_timing(False)
    k_ms = float(np.mean(k_list))
    stage_ms = [a / k_steps for a in stage_acc]
    per_rank = cx.all_values([k_ms] + stage_ms + [0.0] * (5 - len(stage_ms)))
    out = dict(value=value, ms_per_step=dev_ms_max / steps, launches=int(launches), counters=counters, k_ms=k_ms, stage_ms=stage_ms,
               per_rank_kernel_ms=[r[0] for r in per_rank], per_rank_stage_ms=[r[1:1 + len(stage_ms)] for r in per_rank],
               wall_s=t_wall, fused=bool(fused), params=p, idx=idx,
               warmup_note=(f"warm-up steps run on the first {n_warm} pairs of every shard (a full step takes seconds)" if big else None))
    if sampler is not None:
        out["clocks"] = sampler.stop()

    # ---------------- end-to-end arm (host buffers in, host records out) ----------------
    if with_e2e:
        ranges_pin = torch.from_numpy(wl.ranges).pin_memory()
        n_out = n_global if (world > 1 and rank == 0) else len(idx)
        out_pin = torch.empty(max(n_out, 1) * sharded.RECORD_BYTES, dtype=torch.uint8).pin_memory()
        src_l, tgt_l, guess_l = wl.src_idx[idx], wl.tgt_idx[idx], wl.guess[idx]
        used = None
        if world > 1:      # a rank needs only the scans its shard touches: read in place from page-locked memory
            used = shard.plan_subset(wl.src_idx, wl.tgt_idx, wl.n_scans)
            src_e, tgt_e = shard._remap[src_l], shard._remap[tgt_l]
        else:
            src_e, tgt_e = src_l, tgt_l

        def step_e2e():
            if used is None:
                sm.upload_ranges_ptr(ranges_pin.data_ptr(), wl.n_scans, n_beams, wl.scanner)           # H2D + scan->cloud
            else:
                sm.upload_ranges_subset(ranges_pin.data_ptr(), used, wl.scanner, n_scans_total=wl.n_scans, n_beams=n_beams)
            sm.set_pairs(src_e, tgt_e, guess_l)                                                        # H2D pair list
            sm.run(p)
            if world == 1:
                sm.fetch_results_ptr(out_pin.data_ptr(), len(idx))                                     # D2H records (syncs)
            elif fused:
                sm.synchronize()
                cx.dist.barrier()                 # every rank's peer stores have landed
                if rank == 0:
                    sm.gather_fetch_range(0, n_global, host_ptr=out_pin.data_ptr())                    # the WHOLE batch, global order
                cx.dist.barrier()                 # nobody starts the next step's stores into a buffer still being read
            else:
                recv = shard.gather_device()
                if rank == 0:
                    torch.cuda.current_stream().synchronize()
                    host = recv.cpu()             # rank-major; the host interleave is part of this path's cost
                    out_pin[:n_global * sharded.RECORD_BYTES].copy_(torch.from_numpy(
                        sharded.interleave(host.numpy().view(sharded.RESULT_DTYPE), n_global, world).view(np.uint8)))
                cx.dist.barrier()

        for _ in range(0 if big else 3):      # big batches: everything is warm already and one e2e step takes seconds
            step_e2e()
        cx.barrier()
        e2e_steps = 1 if big else max(3, min(2 * steps, 40))      # host-clocked: enough steps that one scheduling hiccup does not show
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step_e2e()
        cx.barrier()
        e2e_s = cx.max_over_ranks(time.perf_counter() - t0)
        n_up = wl.n_scans if used is None else len(used)
        out["e2e"] = {"value": n_global * e2e_steps / e2e_s, "unit": UNIT,
                      "h2d_bytes_per_step": int(4 * n_beams * n_up + 24 * len(idx) + (0 if used is None else 4 * n_up)),
                      "d2h_bytes_per_step": int(sharded.RECORD_BYTES * n_out + 4 * n_up + 4), "steps": e2e_steps,
                      "timing": "host clock around upload+convert+pairs+ICP/cov" +
                                ("+fetch" if world == 1 else "+cross-rank sync+rank 0's copy of the whole gathered batch") +
                                ", max over ranks; byte counts are rank 0's"}
        got = np.frombuffer(out_pin.numpy().tobytes(), dtype=rec_local.dtype)[:n_out]
        mine = got[idx] if (world > 1 and rank == 0) else got
        if world == 1 or rank == 0:
            assert mine.tobytes() == rec_local.tobytes(), "e2e records differ from the resident-arm records"
        # restore the resident state (full store, global scan ids) for the checks below
        shard.use_full_store()
        sm.upload_ranges(wl.ranges, wl.scanner)
        shard.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
        shard.run(p)

    # ---------------- in-run checks ----------------
    checks = {}
    if fused:
        allrec = shard.fused_records()                                                    # whole batch, global order
        assert allrec[idx].tobytes() == rec_local.tobytes(), "fused gather does not hold this rank's records"
        shard.detach_fused_gather()
        if rank == 0:
            # 1 GPU == N GPUs: rank 0 re-aligns a strided sample of the GLOBAL batch alone and compares bit for bit
            sidx = np.linspace(0, n_global - 1, min(n_global, 4096)).astype(np.int64)
            one = sm.submit_pairs(wl.src_idx[sidx], wl.tgt_idx[sidx], wl.guess[sidx], p)
            same = one.tobytes() == allrec[sidx].tobytes()
            checks["one_gpu_equals_gathered"] = {"sample": int(len(sidx)), "bit_equal": bool(same)}
            assert same, "records gathered from N GPUs differ from one GPU running the same pairs"
        cx.barrier()
    out["checks"] = checks
    return out, rec_local


def cpu_baseline_block(wl, p, rec_by_global, n_global, full=True):
    """oracle on this box's host cores over a bounded strided sample of the workload; records compared with the GPU's"""
    pts, off = oracle_clouds(wl.ranges, wl.scanner)
    threads = host_threads()
    cidx = choose_cpu_sample(wl.src_idx[:n_global], wl.tgt_idx[:n_global], wl.guess[:n_global], pts, off, p, threads,
                             target_s=12.0 if full else 2.0)
    dt, used, cref = cpu_sample_run(wl.src_idx, wl.tgt_idx, wl.guess, pts, off, p, cidx, threads)
    got = rec_by_global(cidx)
    same = all(np.array_equal(cref[f], got[f]) for f in ("tx", "ty", "rot_c", "rot_s", "iterations", "status", "n_correspondences", "mse"))
    sidx = cidx[::max(1, len(cidx) // 48)][:48]                  # the reference itself is single-threaded (ros::spin)
    dt1, _, _ = cpu_sample_run(wl.src_idx, wl.tgt_idx, wl.guess, pts, off, p, sidx, 1)
    return {"value": len(cidx) / dt, "unit": UNIT, "cores": used, "kind": "port",
            "single_thread_value": len(sidx) / dt1, "single_thread_sample": f"{len(sidx)} pairs, {dt1:.1f} s",
            "sample": f"{len(cidx)} of {n_global} pairs (evenly strided), {dt:.1f} s, oracle port with exact uniform-grid NN, "
                      f"OpenMP over pairs on {used} threads", "records_equal_gpu": bool(same)}


def latency_block(sm):
    """The two drop-in call shapes as a caller on the latency path sees them (host arrays in, host record out, one call at
    a time), GPU vs the oracle's single thread (the reference is single-threaded): runIcp with the reference's
    defaults (divisor 5, live covariance) and at full resolution; and the online caller's batch — one successive pair +
    the loop-closure candidates of the newest node — through the device-resident form (node table up, enumerate, run,
    records back)."""
    from dpg_slam_b200 import synth
    from dpg_slam_b200._abi import COV_CENSI_CORR, ENUM_ONLINE, Params
    from oracle import oracle_py as O
    out = {}
    # a robot circling a 3 m square in the 10 m x 6 m room, one node per metre: after five laps the newest node's
    # preceding node has ~55 loop-closure candidates within the 5 m gate
    n_nodes = 60
    sc = synth.Scanner()
    side = np.array([[-1.5, -1.5], [1.5, -1.5], [1.5, 1.5], [-1.5, 1.5]])
    rng = np.random.default_rng(11)
    poses = np.zeros((n_nodes, 3))
    for k in range(n_nodes):
        e, f = (k // 3) % 4, (k % 3) / 3.0
        a, b = side[e], side[(e + 1) % 4]
        poses[k, :2] = a + f * (b - a) + rng.normal(0, 0.03, 2)
        poses[k, 2] = np.arctan2(b[1] - a[1], b[0] - a[0]) + rng.normal(0, 0.02)
    ranges = synth.cast_scans(synth.world_room(), poses, sc, 11)
    est = (poses + np.stack([rng.normal(0, 0.03, n_nodes), rng.normal(0, 0.03, n_nodes), rng.normal(0, 0.01, n_nodes)], 1)).astype(np.float32)
    passes = np.zeros(n_nodes, np.int32)
    pts, off = O.clouds_from_ranges(ranges, sc)
    from dpg_slam_b200.scanmatch import relative_guess
    pair_ks = [(k, k - 1) for k in range(1, 25)]
    for tag, p in (("run_icp_default_divisor5_live_cov", Params.defaults()),
                   ("run_icp_divisor1_censi_corr", Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR))):
        g_ms, c_ms = [], []
        for s, t in pair_ks:
            S, T = pts[off[s]:off[s + 1]], pts[off[t]:off[t + 1]]
            g = relative_guess(est[t], est[s])
            sm.run_icp(T, S, g, p)                                             # warm (allocation, module load)
            t0 = time.perf_counter(); _, _, _, r = sm.run_icp(T, S, g, p); g_ms.append(1e3 * (time.perf_counter() - t0))
            t0 = time.perf_counter(); o = O.run_pair(S, T, g, p, fast=1); c_ms.append(1e3 * (time.perf_counter() - t0))
            assert (r.tx, r.ty, r.iterations, r.status) == (o.tx, o.ty, o.iterations, o.status)
        out[tag] = {"gpu_ms_median": float(np.median(g_ms)), "gpu_ms_p90": float(np.percentile(g_ms, 90)),
                    "cpu_oracle_1thread_ms_median": float(np.median(c_ms)), "calls": len(pair_ks)}
    sm.upload_ranges(ranges, sc)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    g_ms, n_batch, rec = [], 0, None
    for rep in range(12):
        t0 = time.perf_counter()
        sm.set_nodes(est, passes)
        n_batch, _ = sm.enumerate_pairs_device(ENUM_ONLINE, 5.0, 2.0)
        sm.run(p)
        rec = sm.fetch_results()
        g_ms.append(1e3 * (time.perf_counter() - t0))
    src, tgt, _ = sm.fetch_pairs()
    t0 = time.perf_counter()
    osrc, otgt = O.enumerate_online(est[:, :2], passes, 5.0, 2.0)
    guess = np.stack([O.relative_guess(est[t, :2], float(est[t, 2]), est[s, :2], float(est[s, 2])) for s, t in zip(osrc, otgt)])
    oref, _ = O.run_batch(pts, off, osrc, otgt, guess, p, fast=1, threads=1)
    c_ms = 1e3 * (time.perf_counter() - t0)
    assert np.array_equal(src, osrc) and np.array_equal(tgt, otgt)
    assert all(np.array_equal(oref[f], rec[f]) for f in ("tx", "ty", "iterations", "status"))
    out["online_update_batch"] = {"pairs": int(n_batch), "nodes": int(n_nodes), "gpu_ms_median": float(np.median(g_ms[2:])),
                                  "cpu_oracle_1thread_ms": float(c_ms), "mean_iterations": float(rec["iterations"].mean()),
                                  "what": "updatePoseGraphObsConstraints shape (dpg_slam.cc:255-300): node table H2D + on-device enumeration "
                                          "+ ICP/cov (reference defaults: divisor 5) + records D2H, scan store resident"}
    return out


# ---- product arm: corridor / loop_closure / dense --------------------------------------------------------------------
def run_product_host_list(args):
    from dpg_slam_b200.scanmatch import ScanMatcher
    cx = Ctx(args)
    torch, world, rank = cx.torch, cx.world, cx.rank
    name = args.workload
    w = WORKLOADS[name]
    n_global = (args.pairs or w["pairs_per_gpu"]) * world if w["scaling"] == "weak" else (args.pairs or w["global_pairs"])
    wl = make_host_workload(name, n_global, rank, world)
    peaks = load_peaks()
    with torch.cuda.stream(cx.stream), ScanMatcher(cx.local) as sm:
        sm.set_stream(cx.stream.cuda_stream)
        sampler = ClockSampler(cx.local)       # started before the warm-up so that nvidia-smi is already sampling when the
        sampler.start()                        # timed region begins; stopped after the kernel-only timing loop
        m, rec_local = measure_host_list(cx, sm, name, args.search, wl, n_global, args.steps, args.warmup, sampler=sampler)
        probe = sm.fp32_probe() if rank == 0 else None
        idx = m["idx"]
        line = None
        if rank == 0:
            counts = (wl.ranges < wl.scanner.range_max).sum(axis=1)
            ns, nt = counts[wl.src_idx[idx]], counts[wl.tgt_idx[idx]]
            roof = roofline_block(name, args.search, m["k_ms"], m["stage_ms"], m["counters"], rec_local, ns, nt, probe, peaks)
            roof["per_rank_kernel_ms"] = m["per_rank_kernel_ms"]
            roof["per_rank_stage_ms"] = m["per_rank_stage_ms"]
            p = m["params"]
            cpu = None
            if not args.no_cpu_baseline:
                if world == 1:
                    cpu = cpu_baseline_block(wl, p, lambda g: rec_local[g], n_global, full=True)
                else:        # N > 1: a small oracle sample of rank 0's own shard, as the in-run parity check only
                    from dpg_slam_b200 import synth  # noqa: F401
                    pts, off = oracle_clouds(wl.ranges, wl.scanner)
                    k = np.linspace(0, len(idx) - 1, min(len(idx), 4 * host_threads())).astype(np.int64)
                    _, _, cref = cpu_sample_run(wl.src_idx, wl.tgt_idx, wl.guess, pts, off, p, idx[k], host_threads())
                    same = all(np.array_equal(cref[f], rec_local[k][f]) for f in ("tx", "ty", "iterations", "status", "n_correspondences", "mse"))
                    m["checks"]["oracle_sample"] = {"sample": int(len(k)), "bit_equal": bool(same)}
                    assert same, "GPU records differ from the CPU oracle on the strided sample"
            if cpu is not None:
                assert cpu["records_equal_gpu"], "GPU records differ from the CPU oracle on the strided sample"
            from dpg_slam_b200._abi import FLAG_CONVERGED
            conv = float(((rec_local["status"] & FLAG_CONVERGED) != 0).mean())
            line = {"metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                    "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic", "config": workload_config(name, world, n_global, args.search,
                                                                                 {"gather": gather_desc(world) if m["fused"] or world == 1 else "NCCL all_gather"}),
                    "e2e": m["e2e"], "gpu_launches": m["launches"], "clocks": m["clocks"], "roofline": roof, "cpu_baseline": cpu,
                    "checks": m["checks"], "wall_s_timed_region": m["wall_s"], "warmup_note": m["warmup_note"],
                    "stats": {"mean_iterations": float(rec_local["iterations"].mean()), "p95_iterations": float(np.percentile(rec_local["iterations"], 95)),
                              "max_iterations": int(rec_local["iterations"].max()), "converged_frac": conv,
                              "distance_evals_per_launch": m["counters"]["distance_evals"], "box_tests_per_launch": m["counters"]["box_tests"]}}
        # the re-alignment shape of this batch (N = 1 default run only): DpgSLAM::reoptimize (dpg_slam.cc:35-120) aligns the same
        # pairs again after every pass, so the previous alignment's iteration counts are known; handed back as cost hints
        # (dpgicp_set_pair_cost_hints) the long alignments start first.  A secondary figure: the headline runs without hints.
        if world == 1 and name == "corridor" and not args.no_also:
            p_h = m["params"]
            sm.upload_ranges(wl.ranges, wl.scanner)
            sm.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
            sm.set_pair_cost_hints(rec_local["iterations"].astype(np.float32))
            for _ in range(3):
                sm.run(p_h)
            h_ms, _ = cx.timed_steps(lambda: sm.run(p_h), args.steps)
            rec_h = sm.fetch_results()
            assert rec_h.tobytes() == rec_local.tobytes(), "records changed with cost hints (they may only change the schedule)"
            sm.set_pair_cost_hints(None)
            # the same batch with the REFERENCE'S OWN settings (parameters.h:402 down-sampling by 5 -> 217 points, the live
            # diagonal covariance of cov.h:572-575): what a drop-in caller that changes nothing runs
            from dpg_slam_b200._abi import Params as _P
            p_ref = _P.defaults()
            for _ in range(3):
                sm.run(p_ref)
            r_ms, _ = cx.timed_steps(lambda: sm.run(p_ref), args.steps)
            rec_r = sm.fetch_results()
            ref_defaults = {"value": n_global * args.steps / (r_ms * 1e-3), "unit": UNIT, "ms_per_step": r_ms / args.steps,
                            "mean_iterations": float(rec_r["iterations"].mean()),
                            "what": "the corridor batch with dpgicp_default_params() = the reference's parameters.h values (divisor 5: "
                                    "217-point clouds, max 500 iterations, reciprocal, live covariance), resident"}
            hinted = {"value": n_global * args.steps / (h_ms * 1e-3), "unit": UNIT, "ms_per_step": h_ms / args.steps,
                      "records_equal_unhinted": True,
                      "what": "the same resident batch re-aligned with the previous alignment's iteration counts as cost hints "
                              "(reoptimize() shape, dpg_slam.cc:35-120): the most expensive quarter of the pairs starts first"}
        # BASELINE configs[2] measured in the same run (N = 1 default run only): the largest single-GPU configuration
        if world == 1 and name == "corridor" and not args.no_also:
            n2 = WORKLOADS["loop_closure"]["pairs_per_gpu"]
            wl2 = make_host_workload("loop_closure", n2)
            m2, rec2 = measure_host_list(cx, sm, "loop_closure", args.search, wl2, n2, max(3, min(args.steps, 5)), 3, with_e2e=True)
            counts2 = (wl2.ranges < wl2.scanner.range_max).sum(axis=1)
            roof2 = roofline_block("loop_closure", args.search, m2["k_ms"], m2["stage_ms"], m2["counters"], rec2,
                                   counts2[wl2.src_idx], counts2[wl2.tgt_idx], probe, peaks)
            pts2, off2 = oracle_clouds(wl2.ranges, wl2.scanner)
            k = np.linspace(0, n2 - 1, 8 * host_threads()).astype(np.int64)
            _, _, cref = cpu_sample_run(wl2.src_idx, wl2.tgt_idx, wl2.guess, pts2, off2, m2["params"], k, host_threads())
            same = all(np.array_equal(cref[f], rec2[k][f]) for f in ("tx", "ty", "iterations", "status", "n_correspondences", "mse"))
            assert same, "loop-closure records differ from the CPU oracle on the strided sample"
            line["also"] = {"loop_closure": {"config": workload_config("loop_closure", 1, n2, args.search), "value": m2["value"], "unit": UNIT,
                                             "ms_per_step": m2["ms_per_step"], "e2e": m2["e2e"],
                                             "roofline": {k_: roof2[k_] for k_ in ("achieved", "peak", "frac", "algorithmic_speedup", "kernel_ms", "stage_ms")},
                                             "oracle_sample_bit_equal": {"sample": int(len(k)), "bit_equal": bool(same)},
                                             "mean_iterations": float(rec2["iterations"].mean())},
                            "corridor_realigned_with_cost_hints": hinted,
                            "corridor_reference_default_params": ref_defaults}
        if world == 1 and rank == 0 and not args.no_latency:
            line["latency"] = latency_block(sm)                  # last: it replaces the scan store
    if args.dump_outputs:                                        # one GPU: rec_local is the whole batch of the last timed step
        keep = dump_sample(len(rec_local))
        dump_records(args.dump_outputs, rec_local[keep], keep)
    if rank == 0:
        print(json.dumps(line), flush=True)
    cx.close()
    return 0


# ---- product arm: multisession (device-enumerated candidate list) ----------------------------------------------------------
def multisession_config(args, world, n_pairs, search):
    w = WORKLOADS["multisession"]
    sps = args.scans_per_session or w["scans_per_session"]
    cfg = workload_config("multisession", world, 0, search,
                          {"sessions": w["sessions"], "scans_per_session": sps, "world_m": args.world_m, "gates_m": [5.0, 2.0],
                           "gather": "none (1 GPU)" if world == 1 else "peer stores from the kernel epilogue into rank 0's buffer (fused, root only)"})
    cfg.pop("global_pairs"); cfg.pop("pairs_per_gpu")      # the pair count is an OUTPUT of the on-device enumeration: reported beside the config
    return cfg


def multisession_nodes(args):
    """Trajectories of all sessions (every rank builds them: cheap, deterministic per session) -> true poses, drifted
    estimates, pass numbers, and the per-session wall segments."""
    import math
    from dpg_slam_b200 import synth
    w = WORKLOADS["multisession"]
    sps = args.scans_per_session or w["scans_per_session"]
    size = args.world_m
    n_boxes = max(6, int(round(300 * (size / 100.0) ** 2)))
    lib = synth._synth()
    poses_all, segs_all = [], []
    for s in range(w["sessions"]):
        rng = np.random.default_rng(w["seed"] * 1000 + s)
        segs = synth.world_office(size, n_boxes, w["seed"], s, 0.05)
        cur = synth._free_poses(segs, size, 1, rng)[0].copy()
        poses = np.empty((sps, 3))
        sp = segs.ctypes.data
        for i in range(sps):
            poses[i] = cur
            for _ in range(50):
                th = cur[2] + rng.uniform(-0.5, 0.5)
                nx, ny = cur[0] + math.cos(th), cur[1] + math.sin(th)
                if 0.5 < nx < size - 0.5 and 0.5 < ny < size - 0.5 and lib.dpgsynth_is_free(sp, segs.shape[0], nx, ny, 0.35) and \
                        not lib.dpgsynth_inside_box(sp, segs.shape[0], nx, ny):
                    cur = np.array([nx, ny, th])
                    break
                cur[2] += rng.uniform(1.0, 2.5)
        poses_all.append(poses)
        segs_all.append(segs)
    poses = np.concatenate(poses_all)
    rng = np.random.default_rng(w["seed"])
    drift = np.stack([rng.normal(0, 0.08, len(poses)), rng.normal(0, 0.08, len(poses)), rng.normal(0, 0.03, len(poses))], axis=1)
    est = (poses + drift).astype(np.float32)
    passes = np.repeat(np.arange(w["sessions"], dtype=np.int32), sps)
    return poses, est, passes, segs_all, sps


def run_product_multisession(args):
    from dpg_slam_b200 import sharded, synth
    from dpg_slam_b200._abi import ENUM_REOPTIMIZE, FLAG_CONVERGED
    from dpg_slam_b200.scanmatch import ScanMatcher, relative_guess
    cx = Ctx(args)
    torch, dist, world, rank = cx.torch, cx.dist, cx.world, cx.rank
    w = WORKLOADS["multisession"]
    p = bench_params("multisession", args.search)
    sc = synth.Scanner(n_beams=w["beams"])
    t_gen0 = time.perf_counter()
    poses, est, passes, segs_all, sps = multisession_nodes(args)
    n_nodes = len(poses)
    # every rank ray-casts the sessions it owns (session s -> rank s % world); the raw ranges are then all-gathered on the
    # devices over NCCL and converted there — the replicated scan store without pushing it N times through one host
    mine = [s for s in range(w["sessions"]) if s % world == rank]
    d_ranges = torch.empty((n_nodes, w["beams"]), dtype=torch.float32, device=cx.dev)
    for s in mine:
        r = synth.cast_scans(segs_all[s], poses[s * sps:(s + 1) * sps], sc, w["seed"] * 1000 + s)
        d_ranges[s * sps:(s + 1) * sps].copy_(torch.from_numpy(r))
    if world > 1:
        for s in range(w["sessions"]):
            dist.broadcast(d_ranges[s * sps:(s + 1) * sps], src=s % world)
    torch.cuda.synchronize(cx.dev)
    t_gen = time.perf_counter() - t_gen0
    peaks = load_peaks()
    line = None
    with torch.cuda.stream(cx.stream), ScanMatcher(cx.local) as sm:
        sm.set_stream(cx.stream.cuda_stream)
        sm.convert_ranges_device(d_ranges.data_ptr(), n_nodes, w["beams"], sc)
        sm.set_nodes(est, passes)
        sm.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, rank, world)                 # warm-up: allocations
        sm.synchronize()
        cx.barrier()
        t0 = time.perf_counter()
        n_total, n_local = sm.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, rank, world)
        sm.synchronize()
        enum_ms = cx.max_over_ranks(1e3 * (time.perf_counter() - t0))
        shard = sharded.ShardedScanMatcher(sm, rank, world, None, cx.dev)
        shard.n_pairs = n_total
        fused = world > 1 and shard.attach_fused_gather(n_total, root_only=True)
        sampler = ClockSampler(cx.local)
        sampler.start()
        # warm-up on a prefix of every shard (a whole step takes tens of seconds at the full size)
        n_warm = min(n_local, 20_000)
        for _ in range(max(args.warmup, 3)):
            sm.run_range(p, 0, n_warm)
        cx.barrier()
        launches0 = sm.last_run_counters()["kernel_launches"]
        sm.enable_stage_timing(True)
        dev_ms, t_wall = cx.timed_steps(lambda: sm.run(p), args.steps)
        stage_ms = sm.last_run_stage_ms()
        sm.enable_stage_timing(False)
        counters = sm.last_run_counters()
        launches = counters["kernel_launches"] - launches0
        dev_ms_max = cx.max_over_ranks(dev_ms)
        value = n_total * args.steps / (dev_ms_max * 1e-3)
        per_rank = cx.all_values([dev_ms / args.steps] + stage_ms + [0.0] * (5 - len(stage_ms)))
        clocks = sampler.stop()
        # records of this shard, streamed through a pinned buffer in slices (also the D2H leg of the e2e arm below)
        CH = 1 << 20
        pin = torch.empty(CH * sharded.RECORD_BYTES, dtype=torch.uint8).pin_memory()

        def stream_records(fetch, n, keep=None, kept=None):
            """keep: sorted record indices to copy into the list kept"""
            it_sum, conv, it_max = 0.0, 0, 0
            for a in range(0, n, CH):
                c = min(CH, n - a)
                fetch(a, c, pin.data_ptr())
                rec = np.frombuffer(pin.numpy(), dtype=sharded.RESULT_DTYPE, count=c)
                it_sum += float(rec["iterations"].sum()); conv += int(((rec["status"] & FLAG_CONVERGED) != 0).sum())
                it_max = max(it_max, int(rec["iterations"].max()))
                if keep is not None:
                    kept.append(rec[keep[np.searchsorted(keep, a):np.searchsorted(keep, a + c)] - a].copy())
            return it_sum, conv, it_max

        keep, kept = (dump_sample(n_local), []) if args.dump_outputs else (None, None)
        it_sum, conv, it_max = stream_records(lambda a, c, ptr: sm.fetch_results_range(a, c, host_ptr=ptr), n_local, keep, kept)
        if args.dump_outputs:                     # one GPU: this rank's list is the whole batch of the last timed step
            dump_records(args.dump_outputs, np.concatenate(kept), keep)

        # ---------------- end-to-end: node table H2D + enumeration on the device + ICP/cov + gather + records D2H ----------------
        e2e_steps = 1
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            sm.set_nodes(est, passes)
            sm.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, rank, world)
            sm.run(p)
            sm.synchronize()
            if world > 1:
                dist.barrier()
            if rank == 0:
                if fused:
                    stream_records(lambda a, c, ptr: sm.gather_fetch_range(a, c, host_ptr=ptr), n_total)
                else:
                    stream_records(lambda a, c, ptr: sm.fetch_results_range(a, c, host_ptr=ptr), n_local)
            if world > 1:
                dist.barrier()
        e2e_s = cx.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": n_total * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(16 * n_nodes),
               "d2h_bytes_per_step": int(sharded.RECORD_BYTES * (n_total if (fused or world == 1) else n_local)), "steps": e2e_steps,
               "timing": "host clock around node table H2D + on-device enumeration + ICP/cov + cross-rank sync + rank 0's streamed copy of "
                         "the whole gathered batch (scan store resident: the scans do not change between reoptimize() calls), max over ranks"}

        # ---------------- in-run checks: a strided sample of the global list, re-aligned by rank 0 alone from HOST-built pairs ----------------
        checks = {}
        n_s = min(n_total, 2048)
        gidx = np.linspace(0, n_total - 1, n_s).astype(np.int64)
        own = gidx[gidx % world == rank]
        lsrc, ltgt, _ = sm.fetch_pairs(int(own.max() // world) + 1) if len(own) else (np.zeros(0, np.int32),) * 3
        mine_pairs = np.stack([lsrc[own // world], ltgt[own // world]], 1) if len(own) else np.zeros((0, 2), np.int32)
        mine_rec = np.concatenate([sm.fetch_results_range(int(k // world), 1) for k in own]) if len(own) else np.zeros(0, sharded.RESULT_DTYPE)
        if world > 1:
            box = [None] * world
            dist.all_gather_object(box, (own, mine_pairs, mine_rec.tobytes()))
        else:
            box = [(own, mine_pairs, mine_rec.tobytes())]
        if fused:
            gathered = np.concatenate([sm.gather_fetch_range(int(k), 1) for k in gidx]) if rank == 0 else None
        if rank == 0:
            order = np.concatenate([b[0] for b in box])
            pairs = np.concatenate([b[1] for b in box])[np.argsort(order)]
            recs = np.concatenate([np.frombuffer(b[2], dtype=sharded.RESULT_DTYPE) for b in box])[np.argsort(order)]
            guess = np.stack([relative_guess(est[t], est[s]) for s, t in pairs])
            one = sm.submit_pairs(pairs[:, 0], pairs[:, 1], guess, p)              # host pair list, one GPU
            same = one.tobytes() == recs.tobytes()
            checks["one_gpu_host_list_equals_sharded_device_list"] = {"sample": int(n_s), "bit_equal": bool(same)}
            assert same, "sharded device-enumerated batch differs from one GPU running the host-built pairs"
            if fused:
                g_same = gathered.tobytes() == recs.tobytes()
                checks["gathered_buffer_holds_every_ranks_records"] = {"sample": int(n_s), "bit_equal": bool(g_same)}
                assert g_same
        if fused:
            shard.detach_fused_gather()

        if rank == 0:
            probe = sm.fp32_probe()
            sm_mhz = float(peaks.get("sm_max_mhz", 1965.0))
            peak32, _, _ = fp32_peak(probe, 148 * 128 * sm_mhz * 1e6 / 1e12)
            k_ms = dev_ms / args.steps
            exec_tflops = (5.0 * counters["distance_evals"] + 9.0 * counters["box_tests"]) / (k_ms * 1e-3) / 1e12
            roof = {"kernel": "dpg::icp_pairs_kernel<WARPS,SEARCH,CLUSTER> (stage chain, rank 0's shard)", "bound": "fp32",
                    "achieved": exec_tflops, "peak": peak32, "unit": "TFLOP/s", "frac": exec_tflops / peak32 if peak32 else None,
                    "achieved_definition": "EXECUTED FP32 work: (5 flop x distance evaluations + 9 flop x box lower bounds) counted on the device / "
                                           "live kernel time (CUDA events on the launching stream)",
                    "peak_source": "dpgicp_fp32_probe / dpgicp_fp32x2_probe in this run (separately rounded multiply+add chains, "
                                   f"scalar and packed alike); nominal {148 * 128 * sm_mhz * 1e6 / 1e12:.1f}",
                    "smem": smem_block(counters, k_ms, sm_mhz),
                    "kernel_ms": k_ms, "stage_ms": stage_ms, "per_rank_kernel_ms": [r[0] for r in per_rank],
                    "per_rank_stage_ms": [r[1:1 + len(stage_ms)] for r in per_rank], "traffic": None,
                    "traffic_source": "not captured for this workload"}
            line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                    "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic", "config": multisession_config(args, world, n_total, args.search),
                    "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": None, "checks": checks,
                    "enumeration": {"nodes": int(n_nodes), "pairs": int(n_total), "pairs_this_rank": int(n_local), "ms": enum_ms,
                                    "what": "count pass + device scan + fill pass incl. every pair's guess, this rank's shard; max over ranks"},
                    "warmup_note": f"warm-up steps run on the first {n_warm} pairs of every shard (a full step takes tens of seconds)",
                    "input_generation_s": t_gen, "wall_s_timed_region": t_wall,
                    "stats": {"mean_iterations": it_sum / max(n_local, 1), "max_iterations": it_max, "converged_frac": conv / max(n_local, 1),
                              "distance_evals_per_launch": counters["distance_evals"], "box_tests_per_launch": counters["box_tests"]}}
            if not args.no_cpu_baseline:
                # oracle on a bounded strided sample of the sampled pairs (clouds rebuilt by the oracle from the same ranges)
                from oracle import oracle_py as O
                k = min(len(pairs), 4 * host_threads())
                sel = np.linspace(0, len(pairs) - 1, k).astype(int)
                scans = np.unique(pairs[sel].ravel())
                remap = {int(s): i for i, s in enumerate(scans)}
                rng_h = d_ranges[torch.from_numpy(scans.astype(np.int64)).to(cx.dev)].cpu().numpy()
                pts, off = O.clouds_from_ranges(rng_h, sc)
                ss = np.array([remap[int(s)] for s in pairs[sel, 0]], np.int32)
                tt = np.array([remap[int(t)] for t in pairs[sel, 1]], np.int32)
                t0 = time.perf_counter()
                cref, used = O.run_batch(pts, off, ss, tt, guess[sel], p, fast=1, threads=host_threads())
                dt = time.perf_counter() - t0
                same = all(np.array_equal(cref[f], recs[sel][f]) for f in ("tx", "ty", "iterations", "status", "n_correspondences", "mse"))
                assert same, "GPU records differ from the CPU oracle on the strided sample"
                line["cpu_baseline"] = {"value": k / dt, "unit": UNIT, "cores": used, "kind": "port",
                                        "sample": f"{k} pairs strided over the whole candidate list, {dt:.1f} s, oracle port, OpenMP over pairs",
                                        "records_equal_gpu": bool(same)}
            print(json.dumps(line), flush=True)
    cx.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the single-call / online-batch latency measurements (N = 1)")
    ap.add_argument("--no-also", action="store_true", help="skip the additional BASELINE configs[2] measurement of the default run")
    ap.add_argument("--workload", default="corridor", choices=sorted(WORKLOADS))
    ap.add_argument("--search", default="pruned", choices=["pruned", "projective"])
    ap.add_argument("--pairs", type=int, default=0, help="override the workload's pair count (per GPU for weak, global for strong scaling)")
    ap.add_argument("--scans-per-session", type=int, default=0, help="multisession: scans per session (default 50000)")
    ap.add_argument("--world-m", type=float, default=100.0, help="multisession: side of the square world in metres")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the records of the last step as DIR/<field>.npy (float32/float64; a "
                         "fixed seeded sample when the batch exceeds 64 MB), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "product" or args.gpus != 1):
        # the reference arm times a sample of pairs sized by a timing pilot: its outputs are not comparable run to run
        ap.error("--dump-outputs needs --impl product and --gpus 1")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "multisession":
        return run_product_multisession(args)
    return run_product_host_list(args)


if __name__ == "__main__":
    sys.exit(main())
