"""Per-update latency of the online caller (updatePoseGraphObsConstraints after each createNode, dpg_slam.cc:255-314,
462-513) on a 2-pass corridor at 1 k / 10 k / 50 k nodes, 1081 beams.  For the newest nodes the scan store is brought up
to date in two ways, alternating in one process (one context each):
  (a) full    upload_ranges of every scan so far (the only way before dpgicp_append_ranges),
  (b) append  append_ranges of the new scan,
each followed by set_nodes -> enumerate_pairs_device(ONLINE) -> run -> records + factors back.  Every step ends in a
device synchronisation, so the host clock around a step is its time.  The records and factors of (a) and (b) must be
equal bit for bit.  Writes one JSON file (default profiles/online_replay.json) with medians and p90 of (a) and (b), the
per-step split, and the card name, power limit and SM clock read in the same run."""
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
from dpg_slam_b200._abi import COV_CENSI_CORR, ENUM_ONLINE, Params  # noqa: E402
from dpg_slam_b200.scanmatch import ScanMatcher  # noqa: E402

STEPS = ("store", "set_nodes", "enumerate_run_fetch")


def card():
    q = ("name", "power.limit", "clocks.sm", "clocks.max.sm")
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={','.join(q)}", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        f = [x.strip() for x in r.stdout.strip().split(",")]
    except OSError:
        f = []
    return dict(zip(q, f)) if len(f) == len(q) else {"nvidia_smi": "unavailable"}


def update(sm, mode, wl, k, p):
    t0 = time.perf_counter()
    if mode == "full":
        sm.upload_ranges(wl.ranges[:k + 1], wl.scanner)
    else:
        sm.append_ranges(wl.ranges[k:k + 1], wl.scanner)
    t1 = time.perf_counter()
    sm.set_nodes(wl.poses_est[:k + 1], wl.passes[:k + 1])
    t2 = time.perf_counter()
    sm.enumerate_pairs_device(ENUM_ONLINE, 5.0, 2.0)
    sm.run(p)
    rec, fac = sm.fetch_results(), sm.fetch_factors()
    t3 = time.perf_counter()
    return (t1 - t0, t2 - t1, t3 - t2), rec, fac


def stats(rows):
    a = 1e3 * np.array(rows)                                   # (updates, steps) in ms
    tot = a.sum(axis=1)
    return {"median_ms": float(np.median(tot)), "p90_ms": float(np.percentile(tot, 90)),
            "split_median_ms": {s: float(np.median(a[:, i])) for i, s in enumerate(STEPS)},
            "split_p90_ms": {s: float(np.percentile(a[:, i], 90)) for i, s in enumerate(STEPS)}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--nodes", default="1000,10000,50000")
    ap.add_argument("--updates", type=int, default=60, help="timed updates per size and configuration")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "online_replay.json"))
    args = ap.parse_args()
    configs = (("reference_defaults_divisor5_live", Params.defaults()),
               ("divisor1_censi_corr", Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)))
    out = {"what": __doc__, "card_before": card(), "updates_timed": args.updates, "warmup_updates": args.warmup,
           "beams": 1081, "passes": 2, "results": []}
    all_equal = True
    for n in (int(x) for x in args.nodes.split(",")):
        wl = synth.config_corridor_passes(n, 1081, 2, seed=2)
        first = n - args.updates - args.warmup
        for tag, p in configs:
            times = {"full": [], "append": []}
            pairs, equal = [], True
            with ScanMatcher(0) as full, ScanMatcher(0) as app:
                app.upload_ranges(wl.ranges[:first], wl.scanner)      # the map so far; the newest nodes are appended
                for i, k in enumerate(range(first, n)):
                    res = {}
                    for mode in (("full", "append") if i % 2 == 0 else ("append", "full")):
                        dt, rec, fac = update(full if mode == "full" else app, mode, wl, k, p)
                        res[mode] = (rec.tobytes(), fac.tobytes())
                        if i >= args.warmup:
                            times[mode].append(dt)
                    equal &= res["full"] == res["append"]
                    pairs.append(len(rec))
            all_equal &= equal
            a, b = stats(times["full"]), stats(times["append"])
            row = {"nodes": n, "config": tag, "pairs_per_update_mean": float(np.mean(pairs)), "full_upload": a, "append": b,
                   "speedup_median": a["median_ms"] / b["median_ms"], "records_and_factors_bit_equal": bool(equal)}
            out["results"].append(row)
            print(json.dumps({k: row[k] for k in ("nodes", "config", "pairs_per_update_mean", "speedup_median",
                                                  "records_and_factors_bit_equal")}),
                  f"full {a['median_ms']:.3f}/{a['p90_ms']:.3f} ms, append {b['median_ms']:.3f}/{b['p90_ms']:.3f} ms "
                  f"split {b['split_median_ms']}", flush=True)
    out["card_after"] = card()
    out["records_and_factors_bit_equal"] = bool(all_equal)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    if not all_equal:
        sys.exit("records of the full-upload and the append paths differ")


if __name__ == "__main__":
    main()
