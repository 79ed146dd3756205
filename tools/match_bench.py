"""Throughput of fe_match_descriptors_device on one GPU: three workloads on device-resident descriptors.

  W1  config 2, 10,000 scans: scan s against scan s-1 (9,999 small groups)
  W2  config 4, 1,000 scans: scan s against scan s-1
  W3  W1's descriptors: the keypoints of the first 1,000 scans against all rows, one group

Each call is timed with CUDA events on the context's stream (fe_timer_begin/end around one call: the work-item
upload, the kernels and the copy of the results); the median of --reps calls after --warmup calls is reported.
Element updates are pairs x 23,760 (12 shifts x 1,980 squared differences); the FP32 issue ceiling is 2 instructions
per element on SMs x 128 lanes x clocks.max.sm read in the same run.  Yardsticks for W3: torch on the GPU (12 rolled
copies + torch.cdist, FP32, not bit-exact) and the CPU oracle on all host cores for a sample of queries.

    python tools/match_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ELEMENTS_PER_PAIR = 12 * 1980


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, plim, clk = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit_w": float(plim), "clocks_max_sm_mhz": float(clk)}


def batch(cfg, n_scans, torch):
    from feature_extraction_b200 import FeatureExtractionNode, node_default, synth
    P = node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    pts, offs, rp = synth.generate(cfg, n_scans)
    npts = int(offs[-1])
    node = FeatureExtractionNode(P, max_points=npts + 4096, max_scans=n_scans,
                                 max_keypoints=max(4096, n_scans * (64 if cfg == 4 else 16)),
                                 max_ring_clusters=max(1 << 20, n_scans * 512))
    d_pts = torch.from_numpy(pts).cuda()
    torch.cuda.synchronize()
    return node, d_pts, offs, rp


def median_ms(node, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        node.timerBegin()
        fn()
        ts.append(node.timerEnd())
    return float(np.median(ts)), ts


def record(name, ms, pairs, clk_mhz, sms, extra=None):
    el = pairs * ELEMENTS_PER_PAIR
    ceiling = 2.0 * el / (sms * 128 * clk_mhz * 1e6)  # seconds at the FP32 issue ceiling
    r = {"workload": name, "ms": round(ms, 4), "pairs": int(pairs), "pairs_per_s": pairs / (ms * 1e-3),
         "element_updates_per_s": el / (ms * 1e-3), "fp32_issue_ceiling_fraction": round(ceiling / (ms * 1e-3), 4)}
    r.update(extra or {})
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scans", type=int, default=10000, help="W1's batch (config 2)")
    ap.add_argument("--scans4", type=int, default=1000, help="W2's batch (config 4)")
    ap.add_argument("--w3-scans", type=int, default=1000, help="W3's queries: the keypoints of this many first scans")
    ap.add_argument("--oracle-queries", type=int, default=32, help="W3 queries the CPU oracle matches")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from match_oracle import binding as mo
    info = card()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    info["sms"] = sms
    clk = info["clocks_max_sm_mhz"]
    print(json.dumps(info), flush=True)
    results = {"card": info, "workloads": []}

    # W1 and W3: config 2
    node, d_pts, offs, rp = batch(2, a.scans, torch)
    step_ms, _ = median_ms(node, lambda: node.processBatchDevice(d_pts.data_ptr(), offs, rp), a.reps, a.warmup)
    ko, K, p_kp, p_d = node.processBatchDevice(d_pts.data_ptr(), offs, rp)
    n = np.diff(ko)
    pairs1 = int((n[1:] * n[:-1]).sum())
    ms1, _ = median_ms(node, lambda: node.matchDescriptorsDevice(p_d, 1980, ko[1:], p_d, 1980, ko[:-1]), a.reps, a.warmup)
    results["workloads"].append(record("W1", ms1, pairs1, clk, sms, {
        "keypoints": int(K), "groups": len(n) - 1, "pipeline_step_ms": round(step_ms, 4),
        "fraction_of_pipeline_step": round(ms1 / step_ms, 4)}))

    nq = int(ko[min(a.w3_scans, len(n))])
    qo, ro = np.array([0, nq]), np.array([0, K])
    ms3, _ = median_ms(node, lambda: node.matchDescriptorsDevice(p_d, 1980, qo, p_d, 1980, ro), a.reps, a.warmup)
    dev3 = node.matchDescriptorsDevice(p_d, 1980, qo, p_d, 1980, ro)
    d_host = node.download(p_d, (K, 1980))
    r3 = {"queries": nq, "refs": int(K)}

    # yardstick 1: torch, 12 rolled copies of the references + cdist, FP32 (not bit-exact)
    Q = torch.from_numpy(d_host[:nq]).cuda()
    R = torch.from_numpy(d_host).cuda()
    Qz, Rz = torch.nan_to_num(Q, nan=1e30), torch.nan_to_num(R, nan=1e30)

    def torch_w3():
        best = None
        for s in range(12):
            Rs = Rz.view(-1, 12, 165).roll(-s, dims=1).reshape(-1, 1980)
            D = torch.cdist(Qz, Rs).square_()
            best = D if best is None else torch.minimum(best, D)
        return best.min(dim=1)
    for _ in range(a.warmup):
        torch_w3()
    ts = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch_w3()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    r3["torch_cdist_ms"] = round(float(np.median(ts)), 3)
    r3["torch_matmul_allow_tf32"] = bool(torch.backends.cuda.matmul.allow_tf32)
    del Q, R, Qz, Rz
    torch.cuda.empty_cache()

    # yardstick 2: the CPU oracle on all host cores, a sample of W3's queries against all rows; and bit-equality there
    threads = len(os.sched_getaffinity(0))
    sample = np.linspace(0, nq - 1, min(a.oracle_queries, nq)).astype(np.int64)
    t0 = time.perf_counter()
    ora = mo.match_descriptors(d_host[sample], d_host, n_threads=threads)
    cpu_s = time.perf_counter() - t0
    same = all(np.array_equal(np.asarray(x)[sample].view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(dev3, ora))
    r3.update({"oracle_threads": threads, "oracle_sample_queries": len(sample), "oracle_pairs_per_s": len(sample) * K / cpu_s,
               "oracle_w3_estimate_s": round(nq * K / (len(sample) * K / cpu_s), 1), "sample_bit_equal_to_oracle": bool(same)})
    results["workloads"].append(record("W3", ms3, nq * int(K), clk, sms, r3))
    node.close()
    del d_pts
    torch.cuda.empty_cache()

    # W2: config 4
    node, d_pts, offs, rp = batch(4, a.scans4, torch)
    step4_ms, _ = median_ms(node, lambda: node.processBatchDevice(d_pts.data_ptr(), offs, rp), a.reps, a.warmup)
    ko, K, p_kp, p_d = node.processBatchDevice(d_pts.data_ptr(), offs, rp)
    n = np.diff(ko)
    pairs2 = int((n[1:] * n[:-1]).sum())
    ms2, _ = median_ms(node, lambda: node.matchDescriptorsDevice(p_d, 1980, ko[1:], p_d, 1980, ko[:-1]), a.reps, a.warmup)
    results["workloads"].append(record("W2", ms2, pairs2, clk, sms, {
        "keypoints": int(K), "groups": len(n) - 1, "pipeline_step_ms": round(step4_ms, 4),
        "fraction_of_pipeline_step": round(ms2 / step4_ms, 4)}))
    node.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
