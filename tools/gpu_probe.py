"""Ad-hoc GPU probe (development aid, not part of the product): smoke + timing sweep of the ICP kernel."""
import os, sys, time, json
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from dpg_slam_b200 import synth
from dpg_slam_b200._abi import Params, COV_CENSI_CORR, COV_REFERENCE_LIVE
from dpg_slam_b200.scanmatch import ScanMatcher
from oracle import oracle_py as O


_STREAM = None


def time_run(sm, p, reps=3):
    global _STREAM
    if _STREAM is None:
        _STREAM = torch.cuda.Stream()      # a real (non-NULL) stream: handle 0 would mean "own stream"
    st = _STREAM
    sm.set_stream(st.cuda_stream)
    sm.run(p); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st); sm.run(p); e1.record(st); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts), float(np.median(ts))


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "corridor"
    n_pairs = int(sys.argv[2]) if len(sys.argv) > 2 else 5000
    torch.cuda.init()
    print(torch.cuda.get_device_name(0), flush=True)
    if which == "corridor":
        wl = synth.config_corridor(n_pairs=n_pairs, seed=2)
    else:
        wl = synth.config_loop_closure(n_pairs=n_pairs, n_scans=2000, seed=3)
    out = {}
    # DPGICP_CHAIN values: target warps per stage, "xC" = the last stage as clusters of C CTAs; "default" = the library's
    for chain in ("default", "2", "4", "8", "16", "2,4", "4,8", "8,16", "2,4,16", "4,8,16", "8,16,16x4"):
        if chain == "default":
            os.environ.pop("DPGICP_CHAIN", None)
        else:
            os.environ["DPGICP_CHAIN"] = chain
        with ScanMatcher(0) as sm:
            sm.upload_ranges(wl.ranges, wl.scanner)
            sm.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
            for search in (1, 0):
                for div in (1, 5):
                    if search == 0 and chain != "default":
                        continue
                    p = Params.defaults(downsample_divisor=div, cov_mode=COV_CENSI_CORR, search=search)
                    try:
                        best, med = time_run(sm, p)
                    except Exception as e:
                        print("ERR", chain, search, div, e, flush=True)
                        continue
                    c = sm.last_run_counters()
                    key = f"chain{chain}_s{search}_d{div}"
                    out[key] = dict(ms=best, med=med, pairs_per_s=wl.n_pairs / best * 1e3, evals=c["distance_evals"],
                                    tests=c["box_tests"])
                    print(key, json.dumps(out[key]), flush=True)
    tag = os.path.basename(os.environ.get("DPGICP_LIBRARY", "default")).replace(".so", "")
    with open(os.path.join(ROOT, "gpurun_out", f"probe_{which}_{n_pairs}_{tag}.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
