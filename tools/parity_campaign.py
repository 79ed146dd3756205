"""Large GPU-vs-oracle parity sweep; prints a markdown summary (and writes it to --out FILE when given).

No whitelist: a descriptor row either meets BASELINE.json's 1e-5 relative bar or is counted as failing.
Beside it the north star's tolerance-boundary report over all ten kinds of include/fe_b200.h: pairs within
1e-6 m of each radius predicate (ring clustering, cross-ring merge, 3DSC support, 3DSC density) and the
decisions within 1e-6 m of the crop box, the ring-window ends, the cluster diameter gate and the 3DSC bin
edges, counted by the device's audit kernels and by the CPU oracle — the two must agree.  Last, the cost of
the report: config 2, 10k scans through fe_process_batch with the report off, radius kinds only, all kinds.

  python tools/parity_campaign.py [SHIFT] [--out FILE]     other SHIFTs = other seeded scenes
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from feature_extraction_b200 import FeatureExtractionNode, synth  # noqa: E402
from boundary_oracle import binding as bo  # noqa: E402
from oracle import oracle_binding as ob  # noqa: E402
from util import to_fe_params  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("shift", type=int, nargs="?", default=0, help="offset of the scan indices (other seeded scenes)")
ap.add_argument("--out", metavar="FILE", help="also write the summary to FILE")
args = ap.parse_args()
SHIFT = args.shift
EPS = 1e-6
cores = len(os.sched_getaffinity(0))
rows, brows = [], []
for cfg, nsc, base in ((1, 400, 5000), (2, 4000, 50000), (3, 160, 7000), (4, 240, 9000)):
    P = ob.launch_playback() if cfg == 1 else ob.node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    pts, offs, rp = synth.generate(cfg, nsc, scan_index_base=base + SHIFT)
    nd = FeatureExtractionNode(to_fe_params(P), max_points=int(offs[-1]) + 4096, max_scans=nsc, max_keypoints=max(4096, nsc * 64))
    t = time.time()
    ko, kp, d = nd.processBatch(pts, offs, rp)
    tg = time.time() - t
    nd.enableBoundaryReportAll(EPS)
    nd.processBatch(pts, offs, rp)
    rep = nd.boundaryReportAll()
    nd.enableBoundaryReport(0.0)
    stats_unordered = 0
    t = time.time()
    ko_o, kp_o, d_o, _ = ob.process_batch(P, pts, offs, rp, mode=1, n_threads=cores)
    tc = time.time() - t
    rep_o = bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=EPS, mode=1, n_threads=cores)
    same_off = bool(np.array_equal(ko, ko_o))
    kp_bits = bool(same_off and np.array_equal(kp.view(np.uint32), kp_o.view(np.uint32)))
    row_exact = (d.view(np.uint32) == d_o.view(np.uint32)).all(axis=1) if same_off else np.zeros(0, bool)
    with np.errstate(invalid="ignore", divide="ignore"):
        rel = np.abs(d.astype(np.float64) - d_o) / np.maximum(np.abs(d_o), 1e-300)
    rel = np.where((d == d_o) | (np.isnan(d) & np.isnan(d_o)), 0, rel).max(axis=1) if same_off else np.zeros(0)
    rows.append((cfg, nsc, int(offs[-1]), len(kp_o), same_off, kp_bits, int(row_exact.sum()), int((~row_exact).sum()),
                 float(rel.max()) if len(rel) else 0.0, int((rel > 1e-5).sum()), tg, tc))
    brows.append((cfg, nsc, bool(np.array_equal(rep, rep_o)), int((rep.sum(1) > 0).sum())) + tuple(int(v) for v in rep.sum(0)) +
                 tuple(int(v) for v in rep_o.sum(0)))
    nd.close()
# cost of the report: config 2, 10k scans, fe_process_batch (host buffers in and out), median of 5 after a warm-up
P = ob.node_default()
pts, offs, rp = synth.generate(2, 10000, scan_index_base=60000)
nd = FeatureExtractionNode(to_fe_params(P), max_points=int(offs[-1]) + 4096, max_scans=10000, max_keypoints=1 << 20)
cost = []
for label, on in (("report off", lambda: nd.enableBoundaryReport(0.0)), ("radius kinds 0-3", lambda: nd.enableBoundaryReport(EPS)),
                  ("all kinds 0-9", lambda: nd.enableBoundaryReportAll(EPS))):
    on()
    nd.processBatch(pts, offs, rp)
    ts = []
    for _ in range(5):
        t = time.time()
        nd.processBatch(pts, offs, rp)
        ts.append(time.time() - t)
    cost.append((label, 1e3 * float(np.median(ts))))
nd.close()
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]
out = ["# Parity campaign (GPU C-ABI vs CPU oracle, KD-tree mode), scan-index shift %d" % SHIFT, "",
       "GPU: %s (name, power limit; read in the same run)" % gpu, "",
       "No whitelist.  Bar: keypoints bit-equal, descriptor values within 1e-5 relative.", "",
       "| config | scans | points | keypoints | counts equal | keypoints bit-equal | descriptor rows bit-equal | rows not bit-equal | max rel err | rows > 1e-5 | GPU s (pageable host) | oracle s (all cores) |",
       "|---|---|---|---|---|---|---|---|---|---|---|---|"]
for r in rows:
    out.append("| %d | %d | %d | %d | %s | %s | %d | %d | %.3g | %d | %.3f | %.2f |" % r)
out += ["", "## Tolerance-boundary report, kinds 0-9 (decisions within %g m of their boundary)" % EPS, "",
        "| config | scans | device == oracle | scans with any | " + " | ".join("device: " + k for k in bo.KIND_NAMES) + " | " +
        " | ".join("oracle: " + k for k in bo.KIND_NAMES) + " |",
        "|" + "---|" * 24]
for r in brows:
    out.append("| " + " | ".join(str(v) for v in r) + " |")
out += ["", "## Cost of the report: config 2, 10,000 scans, fe_process_batch, median of 5 (ms)", "",
        "| report | ms per call |", "|---|---|"] + ["| %s | %.1f |" % c for c in cost]
if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(out) + "\n")
print("\n".join(out))
