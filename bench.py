#!/usr/bin/env python
"""bench.py — scans/sec of the per-scan keypoint pipeline (BASELINE.json metric) on N B200s.

A "step" is one pass of the hot path (reference cloudCallback, src:83-117) over one batch of
synthetic VLP-16 scans: BASELINE.json configs[1] — 10k scans, node_default parameters — per GPU.
The one JSON line also carries, under "configs", the same measurement for BASELINE.json's other
configurations (1 single scan, 3 dense urban, 4 descriptor-heavy: value, e2e, roofline, 1-thread CPU
baseline) and, under "config5", the 100k-scan sweep sharded over the N ranks (strong scaling, host-side
gather inside the timed region, next to a bare pinned H2D copy probe).  `--config C` measures one
configuration alone; `--no-subrecords` keeps the line to the main workload.

  value : whole-job scans/s with the points already resident in HBM (fe_process_batch_device),
          timed with CUDA events on the library's stream, max over ranks.
  e2e   : the same metric through the host-buffer C-ABI call (fe_process_batch): pinned host points
          in, H2D + kernels + D2H of keypoints/descriptors inside the timed region.
  roofline     : the dominant HBM-bound kernel's algorithmic bytes / its CUDA-event time vs measured HBM
                 peak; when a stage bound by FP32 issue or latency takes longer it is named beside it
                 (`largest_kernel_by_time`).  Per-kernel times come from the same number of steps repeated
                 right after the timed region with every stage bracketed by CUDA events on the launching
                 stream (fe_enable_stage_timing).
  cpu_baseline : the CPU oracle (a port of the reference's PCL path, KD-tree mode) on this box's
                 host cores, on a bounded sample of the same workload.

`--impl reference` times that CPU path alone with all host threads (the reference itself needs
ROS + PCL and cannot be built in this image).

`--steps` is the number of timed steps of every measurement in the run (sub-records and config 5 too).
`--dump-outputs DIR` writes what the device-resident path returned in its last timed step of the main
configuration (see dump_outputs) as DIR/<name>.npy; the inputs are seeded, so two builds run with the
same arguments can be compared output for output.

Multi-GPU: scans are independent, so every rank processes its own batch (weak scaling) with no
data-path collective; torch.distributed is only the barrier and the max-over-ranks of the time.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
DIST_TEST_PEAK = 2.65e12  # unfused float distance tests/s of the bare loop on one B200 (tools/microbench/f32x2_bench.cu)
sys.path.insert(0, ROOT)

CONFIG_DESC = {
    1: "config1: single synthetic VLP-16 scan, launch_playback params",
    2: "config2: batch of 10k synthetic VLP-16 scans (16 rings x 1800 azimuth steps), node_default params",
    3: "config3: dense urban scans at 4x azimuth density, node_default params",
    4: "config4: descriptor-heavy (descriptor_radius 5.0, hundreds of poles), node_default params",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=0, help="1-5: that configuration alone; default: config 2 plus sub-records")
    ap.add_argument("--no-subrecords", action="store_true")
    ap.add_argument("--sweep-scans", type=int, default=100000, help="total scans of the config-5 sweep")
    ap.add_argument("--in-process", action="store_true", help="config 5 through fe_multi_process_batch: ONE process, --gpus GPUs")
    ap.add_argument("--scans", type=int, default=0, help="scans per GPU per step (default: the config's batch)")
    ap.add_argument("--cpu-sample", type=int, default=1536, help="scans of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.in_process or args.config == 5):
        ap.error("--dump-outputs writes the device-resident path of configs 1-4")
    return args


def default_scans(cfg):
    return {1: 1, 2: 10000, 3: 2500, 4: 1000, 5: 10000}[cfg]


def oracle_params(ob, cfg):
    P = ob.launch_playback() if cfg == 1 else ob.node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    return P


CONFIG_DESC[5] = "config5: 100k-scan sweep of config-2 scans sharded over the GPUs (scan-parallel, host-side gather)"


def product_params(cfg):
    from feature_extraction_b200 import launch_playback, node_default
    P = launch_playback() if cfg == 1 else node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    return P


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_indices):
        """One poller for ALL GPUs of the job (rank 0 starts it; ranks > 0 pass None): a poller per rank
        multiplies the driver queries without adding information."""
        self.gpus = gpu_indices
        self.rows = []
        self.proc = None

    def start(self):
        if self.gpus is None:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ",".join(str(g) for g in self.gpus), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100" if len(self.gpus) == 1 else "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.gpus is None:
            return None
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "gpus": list(self.gpus)}


def host_threads():
    return len(os.sched_getaffinity(0))


def run_reference(args, rank, world):
    """The reference's CPU path (oracle port, KD-tree mode), all host threads, rank 0 only."""
    if rank != 0:
        return
    from feature_extraction_b200 import synth
    from oracle import oracle_binding as ob
    cfg = args.config or 2
    P = oracle_params(ob, cfg)
    cores = host_threads()
    n = max(8, min(args.cpu_sample, args.scans or default_scans(cfg)))
    pts, offs, rp = synth.generate(cfg, n)
    for _ in range(max(args.warmup, 1)):
        ob.process_batch(P, pts[: offs[min(n, 64)]], offs[: min(n, 64) + 1], rp[: min(n, 64)], mode=1, n_threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ob.process_batch(P, pts, offs, rp, mode=1, n_threads=cores)
    dt = (time.perf_counter() - t0) / args.steps
    v = n / dt
    sample = "%d scans of the workload per step, KD-tree oracle, %d threads scan-parallel" % (n, cores)
    out = {
        "metric": "scans/sec", "value": v, "unit": "scans/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "reference",
        "config": {"workload": CONFIG_DESC[cfg], "scans_per_step": n, "points_per_scan_mean": float(offs[-1]) / n},
        "cpu_baseline": {"value": v, "unit": "scans/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "mpoints_per_s": v * float(offs[-1]) / n / 1e6,
    }
    emit(out)



def stage_bytes(st, desc_len=1980):
    """Algorithmic (compulsory single-pass) bytes of every timed stage for one launch.  ONE table:
    DESIGN.md §5 and BASELINE.md §4 quote these same expressions."""
    N, Ns, Nc, Kf, K, M = (st[k] for k in ("points", "surface_points", "crop_points", "ring_clusters", "keypoints", "neighbours"))
    return {
        "K1 level+crop+ring": 16 * N + 16 * Ns + 20 * Nc,
        "K2 ring clusters": 20 * Nc + 16 * Kf,
        "K3 merge keypoints": 16 * Kf + 16 * K,
        "keypoint CSR": 32 * K,
        "K4a surface grid": 16 * Ns + 16 * st.get("halo_points", Ns),  # read the surface stream, keep the points a keypoint can reach
        "K4b mark neighbours": 16 * M + 4 * M,
        "K4c density": 20 * M,
        "K4d shape context": 20 * M + 4 * desc_len * K,
    }


def survey_bytes(st):
    """SURVEY.md §8d's byte accounting (a global-memory multi-pass design: K2a+K2b+K2c, K4a incl. density,
    K4b incl. the histogram), reported as a second fraction beside the fused design's own bytes."""
    N, Nc, Kf, K, M = (st[k] for k in ("points", "crop_points", "ring_clusters", "keypoints", "neighbours"))
    return {
        "K1": (("K1 level+crop+ring",), 32 * N + 20 * Nc),
        "K2 (K2a+K2b+K2c)": (("K2 ring clusters",), 72 * Nc + 28 * Nc + 20 * Nc + 56 * Kf),
        "K3": (("K3 merge keypoints", "keypoint CSR"), 16 * Kf + 16 * K),
        "K4a (grid+density)": (("K4a surface grid", "K4c density"), 92 * N),
        "K4b (gather+histogram)": (("K4b mark neighbours", "K4d shape context"), 20 * M + 7956 * K),
    }


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class Job:
    """rank / world plumbing shared by the measurements."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def concurrent_min(self, fn, tries):
        """min over `tries` of (max over ranks of fn()), every try started behind a barrier: all ranks really
        run fn at the same time in every try (a per-rank min would pick the try in which the others had finished)."""
        best = None
        for _ in range(tries):
            self.barrier()
            v = self.max_over_ranks(fn())
            best = v if best is None else min(best, v)
        return best

    def sum_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def descriptor_parity(dg, d_o):
    with np.errstate(invalid="ignore", divide="ignore"):
        rel = np.abs(dg.astype(np.float64) - d_o) / np.maximum(np.abs(d_o), 1e-300)
    rel = np.where((dg == d_o) | (np.isnan(dg) & np.isnan(d_o)), 0.0, rel)
    rel = np.where(np.isnan(rel), np.inf, rel)
    rows = rel.max(axis=1) if len(rel) else np.zeros(0)
    return {"keypoints": int(len(dg)), "rows_bit_identical": int((dg.view(np.uint32) == d_o.view(np.uint32)).all(axis=1).sum()),
            "rows_beyond_1e-5": int((rows > 1e-5).sum()), "max_rel_err": float(rows.max()) if len(rows) else 0.0}


DUMP_MAX_BYTES = 64 << 20
DUMP_DESCRIPTOR_ROWS = 4096  # 32 MB of descriptors; a batch of 10k scans has ~37k keypoints (290 MB)


def dump_outputs(out_dir, node, ko, K, p_kp, p_d):
    """What a caller of processBatchDevice receives, copied to the host: keypoint_offsets (B+1,) as
    float64, keypoints (K,4) float32, and the (n,1980) float32 descriptors of `descriptor_rows`: every
    keypoint, or a sample of DUMP_DESCRIPTOR_ROWS of them drawn with a fixed seed when there are more."""
    from feature_extraction_b200.node import DESC_LEN
    arrays = {"keypoint_offsets": ko.astype(np.float64), "keypoints": node.download(p_kp, (K, 4))}
    if p_d:
        rows = np.arange(K)
        if K > DUMP_DESCRIPTOR_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(K, DUMP_DESCRIPTOR_ROWS, replace=False))
        arrays["descriptors"] = node.download(p_d, (K, DESC_LEN))[rows]
        arrays["descriptor_rows"] = rows.astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed %d; use fewer --scans" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(job, cfg, B, steps, warmup, cpu_sample=0, packed=False, dump_dir=None):
    """One configuration on every rank (each its own B scans): device-resident value, per-stage times and
    roofline, e2e through the host entry point, optional 1-thread CPU baseline (rank 0 of a 1-GPU job).
    With `dump_dir`, rank 0 writes the results of its last timed device-resident step there."""
    torch = job.torch
    from feature_extraction_b200 import FeatureExtractionNode, PinnedBuffer, synth
    A = synth.default_azimuth_steps(cfg)
    pin = PinnedBuffer((16 * A * B, 4), np.float32)
    pts, offs, rp = synth.generate(cfg, B, scan_index_base=job.rank * B, out=pin.array)
    npts = int(offs[-1])
    P = product_params(cfg)
    est_kp = max(4096, B * (64 if cfg in (3, 4) else 16))
    dev_node = FeatureExtractionNode(P, device=job.local_rank, max_points=npts + 4096, max_scans=B, max_keypoints=est_kp,
                                     max_ring_clusters=max(1 << 20, B * 512))
    d_pts = torch.empty((max(npts, 1), 4), dtype=torch.float32, device="cuda")
    d_pts[:npts].copy_(torch.from_numpy(pts), non_blocking=False)
    torch.cuda.synchronize()

    # ---- value: device-resident hot path ----
    for _ in range(warmup):
        dev_node.processBatchDevice(d_pts.data_ptr(), offs, rp)
    job.barrier()
    launches = 0
    dev_node.timerBegin()
    t0 = time.perf_counter()
    for _ in range(steps):
        ko, K, p_kp, p_d = dev_node.processBatchDevice(d_pts.data_ptr(), offs, rp)
        launches += dev_node.last_launches
    ev_ms = dev_node.timerEnd()
    job.barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms_step = job.max_over_ranks(ev_ms / steps)
    value = job.world * B / (ms_step * 1e-3)
    if dump_dir and job.rank == 0:
        dump_outputs(dump_dir, dev_node, ko, K, p_kp, p_d)  # before the stage-timing steps overwrite the results
    stats = dev_node.batchStats()
    # Per-kernel durations for the roofline: the same steps repeated right here with the stages serialised
    # (fe_enable_stage_timing) and every stage bracketed by CUDA events on the launching stream.
    stage_acc = {}
    dev_node.enableStageTiming(True)
    dev_node.processBatchDevice(d_pts.data_ptr(), offs, rp)
    dev_node.timerBegin()
    for _ in range(steps):
        dev_node.processBatchDevice(d_pts.data_ptr(), offs, rp)
        for nm, ms in dev_node.stageTimes():
            stage_acc[nm] = stage_acc.get(nm, 0.0) + ms
    serial_ms_step = dev_node.timerEnd() / steps
    dev_node.enableStageTiming(False)
    stage_ms = {k: v / steps for k, v in stage_acc.items()}

    # ---- roofline ----
    peak, peak_src = hbm_peak()
    sb = stage_bytes(stats)
    kernels = {}
    for nm, ms in stage_ms.items():
        gbs = sb.get(nm, 0) / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        kernels[nm] = {"ms": ms, "algorithmic_bytes": sb.get(nm, 0), "gbs": gbs, "frac": gbs / peak}
    # `roofline` describes the dominant HBM-bound kernel: the largest by time of the stages that stream
    # arrays through HBM (K1, K4a).  The other stages are bound by FP32 issue (K4c: the exact unfused
    # distance test) or by latency/issue of per-scan sorting and union-find (K2, K3, K4b, K4d); when one of
    # them is the largest stage by time it is named beside it (`largest_kernel_by_time`) with its own limiter.
    HBM_STAGES = ("K1 level+crop+ring", "K4a surface grid")
    streaming = [k for k in HBM_STAGES if k in stage_ms and k in sb]
    dom = max(streaming, key=stage_ms.get) if streaming else None
    top = max((k for k in stage_ms if k in sb), key=stage_ms.get) if stage_ms else None
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if dom and cfg == 2 and os.path.exists(tpath):
        rec = json.load(open(tpath)).get(dom)
        if rec and rec.get("scans"):
            traffic = rec["dram_bytes_per_launch"] * (B / rec["scans"])
    roofline = None
    if dom:
        tot_ms = max(sum(stage_ms.values()), 1e-9)
        roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
                    "frac": kernels[dom]["frac"], "traffic": traffic, "peak_source": peak_src, "share_of_step": stage_ms[dom] / tot_ms,
                    "selection": "largest HBM-streaming stage by time (K1, K4a)"}
        if top != dom:
            rec = {"kernel": top, "ms": stage_ms[top], "share_of_step": stage_ms[top] / tot_ms, "hbm_frac": kernels[top]["frac"]}
            if top == "K4c density" and stats.get("density_tests"):
                # ceiling: the bare unfused 3-D distance-test loop on this GPU, tools/microbench/f32x2_bench.cu
                rate = stats["density_tests"] / (stage_ms[top] * 1e-3)
                rec.update({"bound": "fp32 issue", "achieved": rate, "peak": DIST_TEST_PEAK, "unit": "distance tests/s",
                            "frac": rate / DIST_TEST_PEAK, "peak_source": "measured, tools/microbench/f32x2_bench.cu (DESIGN.md §6)"})
            else:
                rec["bound"] = "issue/latency (per-scan sorting, union-find, ordered sums)"
            roofline["largest_kernel_by_time"] = rec
        # the second accounting (SURVEY.md §8d bytes) and the whole pipeline's compulsory I/O over the step time
        sv = {}
        for nm, (stages, nbytes) in survey_bytes(stats).items():
            ms = sum(stage_ms.get(x, 0.0) for x in stages)
            if ms > 0:
                sv[nm] = {"ms": ms, "bytes": nbytes, "frac": nbytes / (ms * 1e-3) / 1e9 / peak}
        roofline["survey_8d_accounting"] = sv
        io = 16 * stats["points"] + (16 + 7956) * stats["keypoints"]
        roofline["whole_pipeline"] = {"compulsory_io_bytes": io, "frac": io / (ms_step * 1e-3) / 1e9 / peak}

    # ---- e2e: host buffers through fe_process_batch (H2D + kernels + D2H inside the timed region) ----
    dev_node.close()
    del d_pts
    torch.cuda.empty_cache()
    sub_scans = max(64, min(1024, B))
    sub_pts = int(min(npts + 4096, (npts / max(B, 1)) * sub_scans * 1.5 + 16 * A * 4))
    host_node = FeatureExtractionNode(P, device=job.local_rank, max_points=sub_pts, max_scans=sub_scans,
                                      max_keypoints=max(4096, sub_scans * (64 if cfg in (3, 4) else 16)))
    for _ in range(warmup):
        ko, kp, d = host_node.processBatch(pts, offs, rp, copy=False)
    job.barrier()
    t0 = time.perf_counter()
    e2e_launches = 0
    for _ in range(steps):
        ko, kp, d = host_node.processBatch(pts, offs, rp, copy=False)
        e2e_launches += host_node.last_launches
    torch.cuda.synchronize()
    e2e_ms = job.max_over_ranks((time.perf_counter() - t0) * 1e3 / steps)
    if job.world > 1:
        job.dist.barrier()
    e2e_value = job.world * B / (e2e_ms * 1e-3)
    h2d = npts * 16 + (B + 1) * 12 + B * 36
    d2h = int(len(kp)) * 16 + (0 if d is None else int(len(kp)) * 1980 * 4) + (B + 1) * 4 + 32
    out = {
        "value": value, "unit": "scans/s", "ms_per_step": ms_step, "steps": steps, "warmup": warmup,
        "config": {"workload": CONFIG_DESC[cfg], "scans_per_gpu": B, "points_per_scan_mean": npts / max(B, 1), "input_bytes_per_gpu": npts * 16,
                   "l2": "inputs larger than L2, no flush needed" if npts * 16 > 256e6 else "inputs smaller than L2 (single-scan latency case)",
                   "parallelism": "scan-parallel x%d, no collective" % job.world},
        "mpoints_per_s": value * npts / max(B, 1) / 1e6,
        "wall_ms_per_step": wall_ms / steps,
        "e2e": {"value": e2e_value, "unit": "scans/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "mpoints_per_s": e2e_value * npts / max(B, 1) / 1e6, "sub_batch_scans": sub_scans},
        "gpu_launches": launches, "gpu_launches_e2e": e2e_launches,
        "roofline": roofline, "kernels": kernels, "serial_ms_per_step": serial_ms_step, "work": stats,
    }
    if packed:
        # the same call with packed 12-byte xyz records (the path never reads the input intensity, src:154)
        pin12 = PinnedBuffer((max(npts, 1), 3), np.float32)
        pin12.array[:npts] = pts[:, :3]
        for _ in range(2):
            host_node.processBatchLayout(pin12.array[:npts], 12, 0, 4, 8, offs, rp, copy=False)
        job.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            ko12, kp12, d12 = host_node.processBatchLayout(pin12.array[:npts], 12, 0, 4, 8, offs, rp, copy=False)
        torch.cuda.synchronize()
        e2e12_ms = job.max_over_ranks((time.perf_counter() - t0) * 1e3 / steps)
        same12 = bool(np.array_equal(ko12, ko) and np.array_equal(kp12.view(np.uint32), kp.view(np.uint32)))
        ko, kp, d = host_node.processBatch(pts, offs, rp, copy=False)  # leave the float4 results in place for the checks below
        pin12.free()
        out["e2e_packed_xyz"] = {"value": job.world * B / (e2e12_ms * 1e-3), "unit": "scans/s", "ms_per_step": e2e12_ms,
                                 "h2d_bytes_per_step": npts * 12 + (B + 1) * 12 + B * 36, "same_keypoints_as_float4": same12,
                                 "note": "fe_process_batch_layout with 12-byte xyz records"}
        probe_ms = job.concurrent_min(lambda: host_node.h2dProbe(pts), 3)
        out["h2d_probe"] = {"gbs": job.world * npts * 16 / (probe_ms * 1e-3) / 1e9, "ms": probe_ms,
                            "e2e_over_probe": (npts * 16 / (e2e_ms * 1e-3)) / (npts * 16 / (probe_ms * 1e-3)),
                            "note": "bare cudaMemcpyAsync of the same pinned points, all ranks at once (every try behind a barrier), max over ranks, best of 3"}

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only); doubles as an in-run parity check ----
    if cpu_sample > 0 and job.rank == 0 and job.world == 1:
        from oracle import oracle_binding as ob
        OP = oracle_params(ob, cfg)
        n = max(1, min(cpu_sample, B))
        o2 = offs[: n + 1]
        reps = max(1, cpu_sample // n) if n < cpu_sample else 1  # a single scan is repeated so that the clock sees >= cpu_sample scans
        t0 = time.perf_counter()
        for _ in range(reps):
            ko_o, kp_o, d_o, _ = ob.process_batch(OP, pts, o2, rp[:n], mode=1, n_threads=1)
        dt1 = (time.perf_counter() - t0) / reps
        cores = host_threads()
        t0 = time.perf_counter()
        ob.process_batch(OP, pts, o2, rp[:n], mode=1, n_threads=cores, want_desc=False if cfg == 3 else True)
        dtn = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n / dt1, "unit": "scans/s", "cores": 1, "kind": "port",
                               "sample": "first %d scans of the workload, KD-tree oracle, 1 thread (how the reference runs: ros::spin)" % n}
        if cfg != 3:
            out["cpu_baseline"]["all_cores"] = {"value": n / dtn, "cores": cores}
        same = bool(np.array_equal(ko[: n + 1], ko_o) and np.array_equal(kp[: ko[n]].view(np.uint32), kp_o.view(np.uint32)))
        out["parity_vs_oracle_on_sample"] = same
        if same and d is not None and d_o is not None:
            out["descriptor_parity_on_sample"] = descriptor_parity(d[: ko[n]], d_o)
    host_node.close()
    pin.free()
    torch.cuda.empty_cache()
    return out


def host_mem_available_bytes():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    except Exception:
        pass
    return 0


def measure_sweep(job, total, steps, warmup):
    """BASELINE.json configs[4]: one sweep of `total` config-2 scans split into contiguous shards, one per
    rank (strong scaling).  value: every rank's shard resident in HBM, processed in 10k-scan sub-batches;
    e2e: pinned host shard through fe_process_batch, then the host-side gather of all ranks' results in scan
    order on rank 0 (feature_extraction_b200.sharding.SharedGather) — all inside the timed region."""
    torch = job.torch
    from feature_extraction_b200 import FeatureExtractionNode, PinnedBuffer, synth
    from feature_extraction_b200.sharding import SharedGather, shard_range
    A = synth.default_azimuth_steps(2)
    # bounded by host memory: the whole sweep sits in pinned memory on this box (16 B x ~14k points per scan)
    per_scan = int(16 * A * 0.56)  # mean returns per scan are ~0.485 of the 16 x A rays (dropped no-return rays); 15 % headroom
    avail = host_mem_available_bytes()
    need = total * per_scan * 28  # float4 + packed xyz copies, both pinned
    if avail and need > 0.35 * avail:
        total = int(total * 0.35 * avail / need)
    lo, hi = shard_range(total, job.rank, job.world)
    B = hi - lo
    pin = PinnedBuffer((per_scan * max(B, 1) + 16 * A, 4), np.float32)
    t0 = time.perf_counter()
    pts, offs, rp = synth.generate(2, B, scan_index_base=1_000_000 + lo, out=pin.array,
                                   n_threads=max(1, host_threads() // max(job.world, 1)))
    gen_s = time.perf_counter() - t0
    npts = int(offs[-1])
    P = product_params(2)
    sub = 10000
    sub_max_pts = int(max(offs[min(i + sub, B)] - offs[i] for i in range(0, max(B, 1), sub))) if B else 0
    dev_node = FeatureExtractionNode(P, device=job.local_rank, max_points=sub_max_pts + 4096, max_scans=sub, max_keypoints=max(4096, sub * 16),
                                     max_ring_clusters=max(1 << 20, sub * 512))
    d_pts = torch.empty((max(npts, 1), 4), dtype=torch.float32, device="cuda")
    d_pts[:npts].copy_(torch.from_numpy(pts), non_blocking=False)
    torch.cuda.synchronize()

    def device_pass():
        n = 0
        for i in range(0, B, sub):
            j = min(i + sub, B)
            dev_node.processBatchDevice(d_pts.data_ptr(), offs[i:j + 1], rp[i:j])
            n += dev_node.last_launches
        return n
    for _ in range(warmup):
        device_pass()
    job.barrier()
    dev_node.timerBegin()
    launches = 0
    for _ in range(steps):
        launches += device_pass()
    ev_ms = dev_node.timerEnd()
    job.barrier()
    ms_step = job.max_over_ranks(ev_ms / steps)
    dev_node.close()
    del d_pts
    torch.cuda.empty_cache()

    sub_scans = 1024
    sub_pts = int(min(npts + 4096, (npts / max(B, 1)) * sub_scans * 1.5 + 16 * A * 4))
    host_node = FeatureExtractionNode(P, device=job.local_rank, max_points=sub_pts, max_scans=sub_scans, max_keypoints=max(4096, sub_scans * 16))
    sg = SharedGather()
    res = None
    for _ in range(warmup):
        ko, kp, d = host_node.processBatch(pts, offs, rp, copy=False)
        res = sg.gather(ko, kp, d)
    job.barrier()
    t0 = time.perf_counter()
    t_gather = 0.0
    for _ in range(steps):
        ko, kp, d = host_node.processBatch(pts, offs, rp, copy=False)
        tg = time.perf_counter()
        res = sg.gather(ko, kp, d)
        t_gather += time.perf_counter() - tg
    torch.cuda.synchronize()
    e2e_ms = job.max_over_ranks((time.perf_counter() - t0) * 1e3 / steps)
    gather_ms = job.max_over_ranks(t_gather * 1e3 / steps)
    K_total = int(res[0][-1]) if (job.rank == 0 and res is not None) else 0
    ordered = bool(job.rank != 0 or (len(res[0]) == total + 1 and np.all(np.diff(res[0]) >= 0)))
    # the same with packed 12-byte xyz records
    pin12 = PinnedBuffer((max(npts, 1), 3), np.float32)
    pin12.array[:npts] = pts[:, :3]
    host_node.processBatchLayout(pin12.array[:npts], 12, 0, 4, 8, offs, rp, copy=False)
    job.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        ko, kp, d = host_node.processBatchLayout(pin12.array[:npts], 12, 0, 4, 8, offs, rp, copy=False)
        sg.gather(ko, kp, d)
    torch.cuda.synchronize()
    e2e12_ms = job.max_over_ranks((time.perf_counter() - t0) * 1e3 / steps)
    pin12.free()
    # fabric ceiling: bare pinned H2D copies of every rank's shard at the same time
    probe_ms = job.concurrent_min(lambda: host_node.h2dProbe(pts), 2)
    tot_pts = job.sum_over_ranks(float(npts))
    sg.close()
    host_node.close()
    pin.free()
    torch.cuda.empty_cache()
    probe_gbs = tot_pts * 16 / (probe_ms * 1e-3) / 1e9
    e2e_gbs = tot_pts * 16 / (e2e_ms * 1e-3) / 1e9
    return {
        "workload": CONFIG_DESC[5], "scaling": "strong", "total_scans": total, "scans_per_rank": B, "n_gpus": job.world,
        "steps": steps, "warmup": warmup, "generation_s": gen_s,
        "value": total / (ms_step * 1e-3), "unit": "scans/s", "ms_per_step": ms_step, "mpoints_per_s": tot_pts / (ms_step * 1e-3) / 1e6,
        "e2e": {"value": total / (e2e_ms * 1e-3), "unit": "scans/s", "ms_per_step": e2e_ms, "host_gather_ms_per_step": gather_ms,
                "h2d_bytes_per_step": int(tot_pts * 16), "keypoints_gathered": K_total, "gathered_in_scan_order": ordered,
                "input_gbs": e2e_gbs, "note": "fe_process_batch on every rank's shard + SharedGather of all results on rank 0, timed together; host_gather_ms_per_step is the time inside the gather call, max over ranks: copies plus the wait for the slowest rank at its count exchange"},
        "e2e_packed_xyz": {"value": total / (e2e12_ms * 1e-3), "unit": "scans/s", "ms_per_step": e2e12_ms, "h2d_bytes_per_step": int(tot_pts * 12)},
        "h2d_probe": {"gbs": probe_gbs, "ms": probe_ms, "e2e_over_probe": e2e_gbs / probe_gbs,
                      "note": "bare cudaMemcpyAsync of the same pinned shards, all ranks at once (every try behind a barrier), max over ranks, best of 2"},
        "gpu_launches": launches,
    }


def measure_sweep_in_process(args):
    """config 5 through fe_multi_process_batch: ONE process, a host thread and a context per GPU, results
    concatenated on the host in scan order by the library (inside the timed call)."""
    from feature_extraction_b200 import MultiGpuExtractor, PinnedBuffer, synth
    A = synth.default_azimuth_steps(2)
    total = args.sweep_scans
    per_scan = int(16 * A * 0.56)
    avail = host_mem_available_bytes()
    need = total * per_scan * 16
    if avail and need > 0.35 * avail:
        total = int(total * 0.35 * avail / need)
    pin = PinnedBuffer((per_scan * total + 16 * A, 4), np.float32)
    pts, offs, rp = synth.generate(2, total, scan_index_base=1_000_000, out=pin.array)
    npts = int(offs[-1])
    P = product_params(2)
    G = args.gpus
    sub_scans = 1024
    sub_pts = int((npts / total) * sub_scans * 1.5 + 16 * A * 4)
    m = MultiGpuExtractor(list(range(G)), P, max_points=sub_pts, max_scans=sub_scans, max_keypoints=max(4096, sub_scans * 16))
    for _ in range(max(args.warmup, 1)):
        ko, kp, d = m.processBatch(pts, offs, rp, copy=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ko, kp, d = m.processBatch(pts, offs, rp, copy=False)
    ms = (time.perf_counter() - t0) * 1e3 / args.steps
    m.close()
    pin.free()
    return {"workload": CONFIG_DESC[5], "form": "fe_multi_process_batch, one process", "scaling": "strong", "total_scans": total, "n_gpus": G,
            "steps": args.steps, "warmup": args.warmup, "e2e": {"value": total / (ms * 1e-3), "unit": "scans/s", "ms_per_step": ms,
                                                                 "h2d_bytes_per_step": npts * 16, "keypoints_gathered": int(ko[-1]),
                                                                 "gathered_in_scan_order": bool(np.all(np.diff(ko) >= 0))}}


_RESULT_FD = None


def quiet_stdout():
    """stdout carries exactly one JSON line: whatever libraries print there at C level (NCCL's version
    banner, ...) is sent to stderr for the duration of the run; the result goes to the original fd."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(out):
    line = (json.dumps(out) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, line)


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
        return
    if args.in_process:
        emit({"metric": "scans/sec", "impl": "ours", "config5_in_process": measure_sweep_in_process(args)})
        return

    job = Job(args)
    cfg = args.config or 2
    # clocks / throttle reasons are sampled over the whole run (the device-resident timed region alone is
    # shorter than one nvidia-smi sampling period)
    phys = [g.strip() for g in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if g.strip()]
    job_gpus = [phys[i] if i < len(phys) else i for i in range(job.world)]  # nvidia-smi wants physical indices / UUIDs
    sampler = ClockSampler(job_gpus if job.rank == 0 else None)
    sampler.start()

    if cfg == 5:
        sw = measure_sweep(job, args.sweep_scans, args.steps, max(1, min(args.warmup, 1)))
        clocks = sampler.stop()
        if job.rank == 0:
            out = {"metric": "scans/sec", "value": sw["value"], "unit": "scans/s", "n_gpus": job.world, "steps": sw["steps"], "warmup": sw["warmup"],
                   "ms_per_step": sw["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                   "data": "synthetic", "config": {"workload": sw["workload"], "total_scans": sw["total_scans"], "scans_per_gpu": sw["scans_per_rank"],
                                                   "parallelism": "scan-parallel x%d, host-side gather, no collective" % job.world},
                   "e2e": sw["e2e"], "e2e_packed_xyz": sw["e2e_packed_xyz"], "h2d_probe": sw["h2d_probe"], "gpu_launches": sw["gpu_launches"],
                   "clocks": clocks}
            emit(out)
        if job.world > 1:
            job.dist.destroy_process_group()
        return

    B = args.scans or default_scans(cfg)
    want_cpu = 0 if args.no_cpu_baseline else args.cpu_sample
    m = measure(job, cfg, B, args.steps, args.warmup, cpu_sample=want_cpu, packed=True, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if (args.config or args.no_subrecords) else None
    out = {"metric": "scans/sec", "value": m["value"], "unit": "scans/s", "n_gpus": job.world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    for k in ("config", "mpoints_per_s", "wall_ms_per_step", "e2e", "e2e_packed_xyz", "h2d_probe", "gpu_launches", "gpu_launches_e2e", "roofline",
              "kernels", "serial_ms_per_step", "work", "cpu_baseline", "parity_vs_oracle_on_sample", "descriptor_parity_on_sample"):
        if k in m:
            out[k] = m[k]
    out["kernels_note"] = ("per-stage CUDA-event times of %d extra steps run right after the timed region with the stages serialised "
                           "(fe_enable_stage_timing; %.3f ms per step in that mode)" % (args.steps, m["serial_ms_per_step"]))

    # ---- the other BASELINE.json configurations, in the same run (sub-records) ----
    if not args.config and not args.no_subrecords:
        subs = {}
        for c, wu, cs in ((1, 20, 96), (3, 3, 96), (4, 3, 96)):
            try:
                r = measure(job, c, default_scans(c), args.steps, wu, cpu_sample=(0 if args.no_cpu_baseline else cs))
                for k in ("kernels",):  # keep the line readable: stage times only
                    r[k] = {nm: {"ms": v["ms"], "frac": v["frac"]} for nm, v in r[k].items()}
                subs[str(c)] = r
            except Exception as e:  # a sub-record must never cost the main line
                subs[str(c)] = {"error": repr(e)[:300]}
        out["configs"] = subs
        try:
            out["config5"] = measure_sweep(job, args.sweep_scans, args.steps, 1)
        except Exception as e:
            out["config5"] = {"error": repr(e)[:300]}
        clocks = sampler.stop()
    out["clocks"] = clocks
    if job.rank == 0:
        emit(out)
    if job.world > 1:
        job.dist.destroy_process_group()


if __name__ == "__main__":
    main()
