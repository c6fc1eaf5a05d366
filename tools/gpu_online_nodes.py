"""The node-table step of the online caller: dpgicp_set_nodes (whole table) against dpgicp_update_nodes (changed rows)
on a 2-pass corridor, alternating in one process (one context per way).  Three parts:
  split   dpgicp_set_nodes at 50 000 nodes split by the CUDA runtime calls it makes (torch.profiler, a run of its own):
          host-to-device copies (three pageable cudaMemcpyAsync), kernels + synchronisation (launches and
          cudaStreamSynchronize), and the rest of the call (host loop: finiteness, cosf / sinf, staging, call overhead);
  step    the node step alone at 1 k / 10 k / 50 k / 400 k nodes: set_nodes of the whole table against update_nodes of
          k rows, k = 1 (the appended node), 64 and 4 096 (the recent tail moved, plus the appended node) and all;
          the table grows by one node per step in both ways;
  update  one whole online update (append -> node table -> enumerate ONLINE -> run -> records + factors back) with
          reference defaults at 1 k / 10 k / 50 k nodes, the table brought up to date by set_nodes, by update_nodes of
          the appended node, or by sync_nodes (the Python drop-in: it compares the whole estimate vector with the last
          one sent).  Records and factors must be bit-equal between the ways;
  share   where sync_nodes should fall back to set_nodes: at 50 000 nodes a scattered random share of the nodes moves
          (1 % .. 100 %) and the table is brought up to date by set_nodes, update_nodes of the moved rows, or sync_nodes.
Every timed call ends in a device synchronisation, so the host clock around it is its time.  Medians and p90 in ms;
card name, power limit and SM clock are read in the same run.  Writes profiles/online_nodes.json by default."""
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
from dpg_slam_b200._abi import ENUM_ONLINE, ENUM_REOPTIMIZE, Params  # noqa: E402
from dpg_slam_b200.scanmatch import ScanMatcher  # noqa: E402

F32 = np.float32


def card():
    q = ("name", "power.limit", "clocks.sm", "clocks.max.sm")
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={','.join(q)}", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        f = [x.strip() for x in r.stdout.strip().split(",")]
    except OSError:
        f = []
    return dict(zip(q, f)) if len(f) == len(q) else {"nvidia_smi": "unavailable"}


def ms(v):
    a = 1e3 * np.asarray(v)
    return {"median_ms": float(np.median(a)), "p90_ms": float(np.percentile(a, 90))}


def timed(fn, sm):
    t0 = time.perf_counter()
    fn()
    sm.synchronize()
    return time.perf_counter() - t0


def poses_of(n, seed=2):
    """node estimates of synth.config_corridor_passes(n, passes=2) without casting its scans: 1 m apart, the second pass
    driving back, truth + N(0, 0.05 m; 0.02 rad)"""
    rng = np.random.default_rng(seed)
    per = -(-n // 2)
    s = np.arange(n)
    back = s >= per
    k = s % per
    poses = np.stack([5.0 + np.where(back, per - 1 - k, k), rng.uniform(-0.3, 0.3, n),
                      np.where(back, np.pi, 0.0) + rng.uniform(-0.05, 0.05, n)], 1)
    est = poses + rng.normal(0, [0.05, 0.05, 0.02], (n, 3))
    return est.astype(F32), back.astype(np.int32)


def split(n, calls, warmup):
    import torch
    from torch.profiler import ProfilerActivity, profile
    est, passes = poses_of(n + calls + warmup)
    out = {"nodes": n, "calls": calls}
    with ScanMatcher(0) as sm:
        for k in range(warmup):
            sm.set_nodes(est[:n + k], passes[:n + k])
        wall = []
        for k in range(calls):
            m = n + warmup + k
            wall.append(timed(lambda: sm.set_nodes(est[:m], passes[:m]), sm))
        out["wall"] = ms(wall)
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for k in range(calls):
                m = n + warmup + k
                sm.set_nodes(est[:m], passes[:m])
        per = {}
        for e in prof.key_averages():
            if e.key in ("cudaMemcpyAsync", "cudaLaunchKernel", "cudaStreamSynchronize", "cudaMalloc", "cudaFree"):
                per[e.key] = e.cpu_time_total / 1e3 / calls
        out["runtime_calls_ms_per_call"] = per
        copy = per.get("cudaMemcpyAsync", float("nan"))
        kern = per.get("cudaLaunchKernel", 0.0) + per.get("cudaStreamSynchronize", float("nan"))
        out["split_ms"] = {"host_to_device_copies": copy, "kernels_and_sync": kern,
                           "host_loop_and_rest": out["wall"]["median_ms"] - copy - kern}
        out["note"] = "wall: median without the profiler; the split: runtime-call times under the profiler, per call"
    return out


def step(n, ks, steps, warmup, rng):
    est, passes = poses_of(n + steps + warmup + 1)
    rows = []
    for k in ks:
        cur = est.copy()
        base = n - 1
        t = {"set_nodes": [], "update_nodes": []}
        with ScanMatcher(0) as full, ScanMatcher(0) as upd:
            full.set_nodes(cur[:base], passes[:base])
            upd.set_nodes(cur[:base], passes[:base])
            for i in range(steps + warmup):
                m = base + i + 1                                    # the appended node is m - 1
                kk = m if k == "all" else min(k, m)
                ids = np.arange(m - kk, m, dtype=np.int32)
                cur[ids[:-1]] += F32(1e-3) * rng.standard_normal((len(ids) - 1, 3)).astype(F32)
                ways = {"set_nodes": lambda: full.set_nodes(cur[:m], passes[:m]),
                        "update_nodes": lambda: upd.update_nodes(ids, cur[ids], passes[ids], n_nodes=m)}
                for w in (("set_nodes", "update_nodes") if i % 2 == 0 else ("update_nodes", "set_nodes")):
                    dt = timed(ways[w], full if w == "set_nodes" else upd)
                    if i >= warmup:
                        t[w].append(dt)
            equal = True
            for mode in (ENUM_ONLINE, ENUM_REOPTIMIZE):
                full.enumerate_pairs_device(mode, 5.0, 2.0)
                upd.enumerate_pairs_device(mode, 5.0, 2.0)
                equal &= all(a.tobytes() == b.tobytes() for a, b in zip(full.fetch_pairs(), upd.fetch_pairs()))
        a, b = ms(t["set_nodes"]), ms(t["update_nodes"])
        rows.append({"nodes": n, "changed": k, "set_nodes": a, "update_nodes": b,
                     "speedup_median": a["median_ms"] / b["median_ms"], "tables_bit_equal": bool(equal)})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def update(n, updates, warmup):
    wl = synth.config_corridor_passes(n, 1081, 2, seed=2)
    est, passes = wl.poses_est.astype(F32), wl.passes
    p = Params.defaults()
    first = n - updates - warmup
    ways = ("set_nodes", "update_nodes", "sync_nodes")
    t = {w: [] for w in ways}
    equal = True
    sms = {w: ScanMatcher(0) for w in ways}
    try:
        for w, sm in sms.items():
            sm.upload_ranges(wl.ranges[:first], wl.scanner)
            if w == "sync_nodes":
                sm.sync_nodes(est[:first], passes[:first])
            else:
                sm.set_nodes(est[:first], passes[:first])
        for i, k in enumerate(range(first, n)):
            res = {}
            order = ways[i % 3:] + ways[:i % 3]
            for w in order:
                sm = sms[w]
                t0 = time.perf_counter()
                sm.append_ranges(wl.ranges[k:k + 1], wl.scanner)
                if w == "set_nodes":
                    sm.set_nodes(est[:k + 1], passes[:k + 1])
                elif w == "update_nodes":
                    sm.update_nodes([k], est[k:k + 1], passes[k:k + 1])
                else:
                    sm.sync_nodes(est[:k + 1], passes[:k + 1])
                sm.enumerate_pairs_device(ENUM_ONLINE, 5.0, 2.0)
                sm.run(p)
                rec, fac = sm.fetch_results(), sm.fetch_factors()
                dt = time.perf_counter() - t0
                res[w] = (rec.tobytes(), fac.tobytes())
                if i >= warmup:
                    t[w].append(dt)
            equal &= res["set_nodes"] == res["update_nodes"] == res["sync_nodes"]
    finally:
        for sm in sms.values():
            sm.close()
    row = {"nodes": n, "config": "reference_defaults", **{w: ms(t[w]) for w in ways}, "records_and_factors_bit_equal": bool(equal)}
    print(json.dumps(row), flush=True)
    return row


def share(n, shares, steps, warmup, rng):
    est, passes = poses_of(n)
    rows = []
    for sh in shares:
        cur = est.copy()
        ways = ("set_nodes", "update_nodes", "sync_nodes")
        t = {w: [] for w in ways}
        sms = {w: ScanMatcher(0) for w in ways}
        try:
            for w, sm in sms.items():
                sm.sync_nodes(cur, passes) if w == "sync_nodes" else sm.set_nodes(cur, passes)
            k = max(1, int(round(sh * n)))
            for i in range(steps + warmup):
                ids = np.sort(rng.choice(n, k, replace=False)).astype(np.int32)
                cur[ids] += F32(1e-3) * rng.standard_normal((k, 3)).astype(F32)
                call = {"set_nodes": lambda sm: sm.set_nodes(cur, passes),
                        "update_nodes": lambda sm: sm.update_nodes(ids, cur[ids], passes[ids]),
                        "sync_nodes": lambda sm: sm.sync_nodes(cur, passes)}
                for w in ways[i % 3:] + ways[:i % 3]:
                    dt = timed(lambda: call[w](sms[w]), sms[w])
                    if i >= warmup:
                        t[w].append(dt)
            lists = []
            for sm in sms.values():
                sm.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0)
                lists.append([a.tobytes() for a in sm.fetch_pairs()])
            equal = lists[0] == lists[1] == lists[2]
        finally:
            for sm in sms.values():
                sm.close()
        rows.append({"nodes": n, "share": sh, "changed": k, **{w: ms(t[w]) for w in ways}, "tables_bit_equal": bool(equal)})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--split-nodes", type=int, default=50_000)
    ap.add_argument("--step-nodes", default="1000,10000,50000,400000")
    ap.add_argument("--update-nodes", default="1000,10000,50000")
    ap.add_argument("--parts", default="split,step,update,share")
    ap.add_argument("--steps", type=int, default=60, help="timed calls per size and way")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "online_nodes.json"))
    args = ap.parse_args()
    rng = np.random.default_rng(2)
    out = {"what": __doc__, "card_before": card(), "timed_calls": args.steps, "warmup_calls": args.warmup}
    parts = args.parts.split(",")
    if "split" in parts:
        out["split"] = split(args.split_nodes, args.steps, args.warmup)
        print(json.dumps(out["split"]), flush=True)
    if "step" in parts:
        out["step"] = [r for n in args.step_nodes.split(",")
                       for r in step(int(n), (1, 64, 4096, "all"), args.steps, args.warmup, rng)]
    if "update" in parts:
        out["update"] = [update(int(n), args.steps, args.warmup) for n in args.update_nodes.split(",")]
    if "share" in parts:
        out["share"] = share(50_000, (0.01, 0.1, 0.25, 0.5, 0.75, 1.0), args.steps // 2, args.warmup, rng)
    out["card_after"] = card()
    ok = (all(r["tables_bit_equal"] for r in out.get("step", []) + out.get("share", [])) and
          all(r["records_and_factors_bit_equal"] for r in out.get("update", [])))
    out["all_bit_equal"] = bool(ok)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    if not ok:
        sys.exit("the ways differ")


if __name__ == "__main__":
    main()
