"""Time of fe_register_matches_device on one GPU, beside the match and the pipeline step of the same batch.

  R1  config 4, 50 sequences x 20 scans (synth.generate_poses) in one batch: scan s against scan s-1 (999 groups; the
      49 that pair the last scan of one sequence with the first of the next see two scenes, as at a change of scene)
  R2  config 2, 500 sequences x 20 scans: the same (9,999 groups)
  R3  R1's batch: the last scan of each sequence against the keypoints of its 19 previous scans, moved into its frame by
      the ground truth (50 groups of ~20 x ~400 rows)

Inputs stay on the device: points -> fe_process_batch_device -> fe_match_descriptors_device -> fe_match_device_best ->
fe_register_matches_device.  Each call is timed with CUDA events on the context's stream (fe_timer_begin/end around
one call, its uploads, kernels and result copy included); the median of --reps calls after --warmup calls is reported.
The number to read is registration's share of match + register.  Distance tests = sum over groups of
(hypotheses + 1) * n_q * n_r: the scoring, plus the evaluation of the winner (refinement rounds are not counted).

    python tools/register_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, plim, clk = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit_w": float(plim), "clocks_max_sm_mhz": float(clk)}


def median_ms(node, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        node.timerBegin()
        fn()
        ts.append(node.timerEnd())
    return float(np.median(ts))


def sequences(cfg, n_seq, n_scans=20):
    """n_seq sequences of register_cases.sequence concatenated into one batch -> points, offsets, roll_pitch, poses."""
    from feature_extraction_b200 import synth
    from register_cases import sequence
    P, O, RP, POS = [], [0], [], []
    for i in range(n_seq):
        pts, offs, rp, poses = sequence(synth, cfg, i, n_scans)
        P.append(pts)
        O.extend(O[-1] + offs[1:])
        RP.append(rp)
        POS.append(poses)
    return np.concatenate(P), np.array(O, np.int64), np.concatenate(RP), POS


def tests_of(qo, ro, nhyp):
    nq, nr = np.diff(qo), np.diff(ro)
    return int(((nhyp.astype(np.int64) + 1) * nq * nr).sum())


def run(name, cfg, n_seq, a, torch, results, submap=False):
    from feature_extraction_b200 import FeatureExtractionNode, node_default, register_params_default
    from register_cases import apply
    P = node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    pts, offs, rp, poses = sequences(cfg, n_seq)
    B = len(offs) - 1
    node = FeatureExtractionNode(P, max_points=int(offs[-1]) + 4096, max_scans=B,
                                 max_keypoints=max(4096, B * (64 if cfg == 4 else 16)), max_ring_clusters=max(1 << 20, B * 512))
    d_pts = torch.from_numpy(pts).cuda()
    torch.cuda.synchronize()
    step = median_ms(node, lambda: node.processBatchDevice(d_pts.data_ptr(), offs, rp), a.reps, a.warmup)
    ko, K, p_kp, p_d = node.processBatchDevice(d_pts.data_ptr(), offs, rp)
    prm = register_params_default()
    keep = []
    if not submap:  # scan s against s-1 of the batch; 1 group in 20 pairs two sequences (a change of scene)
        qo, ro = ko[1:], ko[:-1]
        qp, rp_, dq, dr = p_kp, p_kp, p_d, p_d
        groups = B - 1
    else:  # the last scan of each sequence against its 19 predecessors, moved into its frame
        kp = node.download(p_kp, (K, 4))
        d = node.download(p_d, (K, 1980))
        Q, R, Dq, Dr, qo, ro = [], [], [], [], [0], [0]
        for i in range(n_seq):
            s = 20 * i + 19
            pz = poses[i]
            c, si, x, y = np.cos(pz[19, 2]), np.sin(pz[19, 2]), pz[19, 0], pz[19, 1]
            Q.append(kp[ko[s]:ko[s + 1]])
            Dq.append(d[ko[s]:ko[s + 1]])
            for t in range(19):
                rows = kp[ko[20 * i + t]:ko[20 * i + t + 1]].copy()
                w = np.array([np.cos(pz[t, 2]), np.sin(pz[t, 2]), pz[t, 0], pz[t, 1]])
                xy = apply(w, rows[:, :2]) - [x, y]
                rows[:, 0], rows[:, 1] = c * xy[:, 0] + si * xy[:, 1], -si * xy[:, 0] + c * xy[:, 1]
                R.append(rows)
                Dr.append(d[ko[20 * i + t]:ko[20 * i + t + 1]])
            qo.append(qo[-1] + len(Q[-1]))
            ro.append(sum(len(x) for x in R))
        qo, ro = np.array(qo), np.array(ro)
        tq, tr = torch.from_numpy(np.concatenate(Q)).cuda(), torch.from_numpy(np.concatenate(R).astype(np.float32)).cuda()
        tdq, tdr = torch.from_numpy(np.concatenate(Dq)).cuda(), torch.from_numpy(np.concatenate(Dr)).cuda()
        keep = [tq, tr, tdq, tdr]
        torch.cuda.synchronize()
        qp, rp_, dq, dr = tq.data_ptr(), tr.data_ptr(), tdq.data_ptr(), tdr.data_ptr()
        groups = n_seq
    match = median_ms(node, lambda: node.matchDescriptorsDevice(dq, 1980, qo, dr, 1980, ro), a.reps, a.warmup)
    node.matchDescriptorsDevice(dq, 1980, qo, dr, 1980, ro)
    p_best = node.matchDeviceBest()
    reg = median_ms(node, lambda: node.registerMatchesDevice(qp, rp_, p_best, qo, ro, prm), a.reps, a.warmup)
    out = node.registerMatchesDevice(qp, rp_, p_best, qo, ro, prm)
    r = {"workload": name, "config": cfg, "scans": B, "keypoints": int(K), "groups": int(groups),
         "query_rows": int(qo[-1] - qo[0]), "ref_rows_max_group": int(np.diff(ro).max()),
         "hypotheses": int(out["n_hypotheses"].sum()), "distance_tests": tests_of(qo, ro, out["n_hypotheses"]),
         "registered_fraction": round(float((out["status"] == 2).mean()), 4),
         "pipeline_step_ms": round(step, 4), "match_ms": round(match, 4), "register_ms": round(reg, 4),
         "register_share_of_match_plus_register": round(reg / (match + reg), 4),
         "register_fraction_of_pipeline_step": round(reg / step, 4)}
    print(json.dumps(r), flush=True)
    results["workloads"].append(r)
    node.close()
    del d_pts, keep
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seq4", type=int, default=50, help="R1 / R3 sequences of 20 scans (config 4)")
    ap.add_argument("--seq2", type=int, default=500, help="R2 sequences of 20 scans (config 2)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    info = card()
    info["sms"] = torch.cuda.get_device_properties(0).multi_processor_count
    print(json.dumps(info), flush=True)
    results = {"card": info, "workloads": []}
    run("R1", 4, a.seq4, a, torch, results)
    run("R2", 2, a.seq2, a, torch, results)
    run("R3", 4, a.seq4, a, torch, results, submap=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
