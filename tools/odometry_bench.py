"""Time of fe_odometry_device on one GPU, beside the match and the scan-against-scan registration of the same batch.

  O1  config 4, 50 sequences x 20 scans in one batch (register_bench.py's R1): odometry at the default window and at
      W = 1, beside R1's match and register calls
  O2  config 2, 500 sequences x 20 scans (R2's batch): the same
  O3  config 4, one sequence of --long scans on a path that swings through the pole lattice: the serial case, where
      three launches per step set the floor

Inputs stay on the device: points -> fe_process_batch_device -> fe_match_descriptors_device (scan s against s-1) ->
fe_match_device_best -> fe_odometry_device.  Each call is timed with CUDA events on the context's stream (fe_timer_begin
/ end around one call, its table upload, kernels and result copy included); the median of --reps calls after --warmup
calls is reported, with the kernel launches of one call.

    python tools/odometry_bench.py [--out FILE.json]
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

from register_bench import card, median_ms, sequences  # noqa: E402


def long_sequence(cfg, n):
    """One path of n scans through the scene of scan 1000 of config cfg, swinging along the lattice (0.4 m a scan)."""
    from feature_extraction_b200 import synth
    s = np.arange(n)
    poses = np.stack([35.0 + 25.0 * np.sin(2 * np.pi * s / 400.0), 3.0 * np.sin(2 * np.pi * s / 100.0),
                      0.05 * np.sin(2 * np.pi * s / 150.0)], axis=1)
    pts, offs, rp = synth.generate_poses(cfg, 1000, poses)
    return pts, offs, rp


def run(name, cfg, pts, offs, rp, so, windows, a, torch, results):
    from feature_extraction_b200 import FeatureExtractionNode, node_default, register_params_default
    P = node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    B = len(offs) - 1
    node = FeatureExtractionNode(P, max_points=int(offs[-1]) + 4096, max_scans=B,
                                 max_keypoints=max(4096, B * (64 if cfg == 4 else 16)), max_ring_clusters=max(1 << 20, B * 512))
    d_pts = torch.from_numpy(pts).cuda()
    torch.cuda.synchronize()
    ko, K, p_kp, p_d = node.processBatchDevice(d_pts.data_ptr(), offs, rp)
    qo, ro = ko[1:], ko[:-1]
    prm = register_params_default()
    match = median_ms(node, lambda: node.matchDescriptorsDevice(p_d, 1980, qo, p_d, 1980, ro), a.reps, a.warmup)
    node.matchDescriptorsDevice(p_d, 1980, qo, p_d, 1980, ro)
    p_best = node.matchDeviceBest()
    reg = median_ms(node, lambda: node.registerMatchesDevice(p_kp, p_kp, p_best, qo, ro, prm), a.reps, a.warmup)
    r = {"workload": name, "config": cfg, "scans": B, "sequences": len(so) - 1, "longest_sequence": int(np.diff(so).max()),
         "keypoints": int(K), "match_ms": round(match, 4), "register_scan_to_scan_ms": round(reg, 4), "odometry": []}
    for W in windows:
        odo = median_ms(node, lambda: node.odometryDevice(p_kp, ko, p_best, so, W, prm), a.reps, a.warmup)
        out = node.odometryDevice(p_kp, ko, p_best, so, W, prm)
        links = out["source"] != 0
        r["odometry"].append({"window": W, "odometry_ms": round(odo, 4), "launches": node.last_launches,
                              "registered_fraction": round(float((out["source"][links] == 1).mean()), 4) if links.any() else None,
                              "hypotheses": int(out["n_hypotheses"].sum())})
    print(json.dumps(r), flush=True)
    results["workloads"].append(r)
    node.close()
    del d_pts
    torch.cuda.empty_cache()


def main():
    from feature_extraction_b200 import ODOMETRY_WINDOW
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seq4", type=int, default=50, help="O1 sequences of 20 scans (config 4)")
    ap.add_argument("--seq2", type=int, default=500, help="O2 sequences of 20 scans (config 2)")
    ap.add_argument("--long", type=int, default=400, help="O3 scans in one config-4 sequence")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    info = card()
    info["sms"] = torch.cuda.get_device_properties(0).multi_processor_count
    print(json.dumps(info), flush=True)
    results = {"card": info, "default_window": ODOMETRY_WINDOW, "workloads": []}
    windows = sorted({ODOMETRY_WINDOW, 1})
    for name, cfg, n in (("O1", 4, a.seq4), ("O2", 2, a.seq2)):
        pts, offs, rp, _ = sequences(cfg, n)
        run(name, cfg, pts, offs, rp, np.arange(0, 20 * n + 1, 20), windows, a, torch, results)
    pts, offs, rp = long_sequence(4, a.long)
    run("O3", 4, pts, offs, rp, np.array([0, a.long]), windows, a, torch, results)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
