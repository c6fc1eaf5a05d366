"""Sustained throughput with several pair batches in flight on one context (batch slots, dpgicp_slot_*).

Workloads, each a sequence of batches with distinct seeds held in ONE scan store:
  corridor      24 batches of 5000 successive pairs x 1081 beams (the bench's corridor batch, seeds 100..123)
  loop_closure   4 batches of 100 000 loop-closure candidates over 2000 scans x 1081 beams (seeds 200..203)
both with divisor 1 and CENSI_CORR covariance.  Every batch sequence is run with 1, 2 and 3 batches in flight (1 = the
default slot: set_pairs -> run -> fetch, one batch at a time; K > 1 = K slots, batch b on slot b % K, launched once that
slot's previous batch is fetched), the modes alternating in rounds after a warm-up round.  Reported per mode: sustained
pairs/s (host clock from the first set_pairs to the last fetch, which ends in a device synchronisation), median and p90
of the per-batch latency (set_pairs -> its records on the host).  Records must be bit-equal across the modes.  The card
name, power limit and SM clock are read in the same run.  Writes one JSON file."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dpg_slam_b200 import synth  # noqa: E402
from dpg_slam_b200._abi import COV_CENSI_CORR, RESULT_DTYPE, Params  # noqa: E402
from dpg_slam_b200.scanmatch import ScanMatcher  # noqa: E402

MODES = (1, 2, 3)


def card():
    q = ("name", "power.limit", "clocks.sm", "clocks.max.sm")
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={','.join(q)}", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        f = [x.strip() for x in r.stdout.strip().split(",")]
    except OSError:
        f = []
    return dict(zip(q, f)) if len(f) == len(q) else {"nvidia_smi": "unavailable"}


def make_batches(name, n_batches, n_pairs):
    """ranges of every batch back to back (one store) and each batch's (src, tgt, guess) into it"""
    ranges, batches, base, scanner = [], [], 0, None
    for b in range(n_batches):
        if name == "corridor":
            wl = synth.config_corridor(n_pairs=n_pairs, n_beams=1081, seed=100 + b)
        else:
            wl = synth.config_loop_closure(n_pairs=n_pairs, n_scans=2000, n_beams=1081, seed=200 + b)
        ranges.append(wl.ranges)
        batches.append((wl.src_idx + base, wl.tgt_idx + base, wl.guess))
        base += wl.n_scans
        scanner = wl.scanner
    return np.concatenate(ranges), scanner, batches


def run_mode(sm, slots, batches, p, recs):
    """all batches with len(slots) in flight; recs[b] receives batch b's records; returns (seconds, latencies)"""
    K = len(slots)
    pending = [None] * K
    lat = []

    def fetch(k):
        b, t_set = pending[k]
        slots[k].fetch_results(len(batches[b][0]), out=recs[b])
        lat.append(time.perf_counter() - t_set)
        pending[k] = None

    t0 = time.perf_counter()
    for b, (s, t, g) in enumerate(batches):
        k = b % K
        if pending[k] is not None:
            fetch(k)
        t_set = time.perf_counter()
        slots[k].set_pairs(s, t, g)
        slots[k].run(p)
        pending[k] = (b, t_set)
    for j in range(K):                       # the oldest batch first
        k = (len(batches) + j) % K
        if pending[k] is not None:
            fetch(k)
    return time.perf_counter() - t0, lat


def measure(name, n_batches, n_pairs, rounds):
    ranges, scanner, batches = make_batches(name, n_batches, n_pairs)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    n_total = sum(len(b[0]) for b in batches)
    sm = ScanMatcher(0)
    sm.upload_ranges(ranges, scanner)
    slots = {K: [sm] if K == 1 else [sm.slot() for _ in range(K)] for K in MODES}
    recs = {K: [np.zeros(len(b[0]), RESULT_DTYPE) for b in batches] for K in MODES}
    times = {K: [] for K in MODES}
    lats = {K: [] for K in MODES}
    for r in range(rounds + 1):              # round 0 warms every shape up and is not kept
        for K in MODES[r % len(MODES):] + MODES[:r % len(MODES)]:
            dt, lat = run_mode(sm, slots[K], batches, p, recs[K])
            if r > 0:
                times[K].append(dt)
                lats[K].extend(lat)
    sm.close()
    ref = b"".join(x.tobytes() for x in recs[1])
    out = {"batches": n_batches, "pairs_per_batch": n_pairs, "rounds": rounds,
           "records_bit_equal_to_one_in_flight": {str(K): b"".join(x.tobytes() for x in recs[K]) == ref for K in MODES},
           "iterations_mean": float(np.mean(np.concatenate([x["iterations"] for x in recs[1]]))), "in_flight": {}}
    for K in MODES:
        t = np.array(times[K])
        lat = np.array(lats[K]) * 1e3
        out["in_flight"][str(K)] = {
            "sustained_pairs_per_s_median": float(n_total / np.median(t)),
            "sustained_pairs_per_s_each_round": [float(n_total / x) for x in t],
            "batch_latency_ms_median": float(np.median(lat)), "batch_latency_ms_p90": float(np.percentile(lat, 90))}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "inflight.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--corridor-batches", type=int, default=24)
    ap.add_argument("--loop-batches", type=int, default=4)
    ap.add_argument("--skip-loop", action="store_true")
    a = ap.parse_args()
    res = {"what": __doc__, "card_before": card()}
    res["corridor"] = measure("corridor", a.corridor_batches, 5000, a.rounds)
    print(json.dumps({"corridor": res["corridor"]["in_flight"]}, indent=1), flush=True)
    if not a.skip_loop:
        res["loop_closure"] = measure("loop_closure", a.loop_batches, 100_000, max(2, a.rounds // 2))
        print(json.dumps({"loop_closure": res["loop_closure"]["in_flight"]}, indent=1), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"equal": {k: res[k]["records_bit_equal_to_one_in_flight"] for k in ("corridor", "loop_closure") if k in res},
                      "card": res["card_before"]}))


if __name__ == "__main__":
    main()
