"""Time of fe_loop_closures_device on one GPU, beside the match and odometry of the same batch.

  L1  config 4, 50 out-and-back sequences of 30 scans (tests/loop_cases.py) in one batch
  L2  config 4, one sequence of --long scans (odometry_bench.py's O3 path): the quadratic retrieval at its largest
  L3  config 2, 500 sequences x 20 scans (register_bench.py's R2 batch)

Inputs stay on the device: points -> fe_process_batch_device -> fe_loop_closures_device, default loop and
registration parameters.  Each call is timed with CUDA events on the context's stream (fe_timer_begin / end around one
call: table upload, kernels and result copy); the median of --reps calls after --warmup calls is reported, with the
kernel launches of one call.  Retrieval and verification are split by a torch.profiler run of its own: the kernels of
one call in launch order, the first k_match_tiles (and its k_match_merge) being retrieval and the rest verification.
Retrieval pairs (sum over eligible scans of n_t x database rows) and element updates (pairs x 23,760) are computed
from the shapes; the FP32 issue ceiling is 2 instructions per element on SMs x 128 lanes at clocks.max.sm (DESIGN.md
§12).  Beside them: the match of scan s against s - 1 and odometry at the default window on the same batch.

    python tools/loop_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from odometry_bench import long_sequence  # noqa: E402
from register_bench import card, median_ms, sequences  # noqa: E402

ELEMENTS = 12 * 12 * 165  # element updates per descriptor pair


def loop_sequences(cfg, n_seq):
    """n_seq out-and-back sequences of loop_cases concatenated into one batch -> points, offsets, roll_pitch."""
    from feature_extraction_b200 import synth
    from loop_cases import loop_sequence
    P, O, RP = [], [0], []
    for i in range(n_seq):
        pts, offs, rp, _ = loop_sequence(synth, cfg, i)
        P.append(pts)
        O.extend(O[-1] + offs[1:])
        RP.append(rp)
    return np.concatenate(P), np.array(O, np.int64), np.concatenate(RP)


def retrieval_pairs(ko, so, gap):
    pairs = 0
    for q in range(len(so) - 1):
        f = so[q]
        for s in range(f + gap, so[q + 1]):
            pairs += int(ko[s + 1] - ko[s]) * int(ko[s - gap + 1] - ko[f])
    return pairs


def split_ms(node, fn, torch):
    """Retrieval and verification kernel time (ms) of one call from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ks = sorted((e for e in prof.events() if e.device_type.name == "CUDA" and "k_" in e.name and "Memcpy" not in e.name),
                key=lambda e: e.time_range.start)
    retrieval, verification, seen_vote = 0.0, 0.0, False
    for e in ks:
        seen_vote |= "k_loop_" in e.name
        if seen_vote:
            verification += e.time_range.elapsed_us() / 1e3
        else:
            retrieval += e.time_range.elapsed_us() / 1e3
    return retrieval, verification, [e.name.split("(")[0] for e in ks]


def run(name, cfg, pts, offs, rp, so, a, torch, info, results):
    from feature_extraction_b200 import (FeatureExtractionNode, ODOMETRY_WINDOW, loop_params_default, node_default,
                                         register_params_default)
    P = node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    B = len(offs) - 1
    node = FeatureExtractionNode(P, max_points=int(offs[-1]) + 4096, max_scans=B,
                                 max_keypoints=max(4096, B * (64 if cfg == 4 else 16)), max_ring_clusters=max(1 << 20, B * 512))
    d_pts = torch.from_numpy(pts).cuda()
    torch.cuda.synchronize()
    ko, K, p_kp, p_d = node.processBatchDevice(d_pts.data_ptr(), offs, rp)
    lp, prm = loop_params_default(), register_params_default()
    call = lambda: node.loopClosuresDevice(p_kp, p_d, 1980, ko, so, lp, prm)  # noqa: E731
    loop_ms = median_ms(node, call, a.reps, a.warmup)
    out = call()
    launches = node.last_launches
    ret, ver, kernels = split_ms(node, call, torch)
    qo, ro = ko[1:], ko[:-1]
    match = median_ms(node, lambda: node.matchDescriptorsDevice(p_d, 1980, qo, p_d, 1980, ro), a.reps, a.warmup)
    node.matchDescriptorsDevice(p_d, 1980, qo, p_d, 1980, ro)
    p_best = node.matchDeviceBest()
    odo = median_ms(node, lambda: node.odometryDevice(p_kp, ko, p_best, so, ODOMETRY_WINDOW, prm), a.reps, a.warmup)
    pairs = retrieval_pairs(ko, so, lp.min_gap)
    ceiling = info["sms"] * 128 * info["clocks_max_sm_mhz"] * 1e6 / 2.0
    rate = pairs * ELEMENTS / (ret / 1e3) if ret > 0 else None
    r = {"workload": name, "config": cfg, "scans": B, "sequences": len(so) - 1, "longest_sequence": int(np.diff(so).max()),
         "keypoints": int(K), "min_gap": lp.min_gap, "candidates": lp.candidates, "loop_ms": round(loop_ms, 4),
         "launches": launches, "kernels": kernels, "retrieval_kernel_ms": round(ret, 4),
         "verification_kernel_ms": round(ver, 4), "retrieval_pairs": pairs, "retrieval_element_updates": pairs * ELEMENTS,
         "retrieval_element_updates_per_s": rate, "of_fp32_issue_ceiling": round(rate / ceiling, 3) if rate else None,
         "loops": int((out["loop"] >= 0).sum()), "match_s_vs_prev_ms": round(match, 4),
         "odometry_default_window_ms": round(odo, 4)}
    print(json.dumps(r), flush=True)
    results["workloads"].append(r)
    node.close()
    del d_pts
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seq4", type=int, default=50, help="L1 out-and-back sequences of 30 scans (config 4)")
    ap.add_argument("--long", type=int, default=400, help="L2 scans in one config-4 sequence")
    ap.add_argument("--seq2", type=int, default=500, help="L3 sequences of 20 scans (config 2)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    info = card()
    info["sms"] = torch.cuda.get_device_properties(0).multi_processor_count
    print(json.dumps(info), flush=True)
    results = {"card": info, "workloads": []}
    pts, offs, rp = loop_sequences(4, a.seq4)
    run("L1", 4, pts, offs, rp, np.arange(0, 30 * a.seq4 + 1, 30), a, torch, info, results)
    pts, offs, rp = long_sequence(4, a.long)
    run("L2", 4, pts, offs, rp, np.array([0, a.long]), a, torch, info, results)
    pts, offs, rp, _ = sequences(2, a.seq2)
    run("L3", 2, pts, offs, rp, np.arange(0, 20 * a.seq2 + 1, 20), a, torch, info, results)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
