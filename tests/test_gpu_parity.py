"""Parity of the CUDA path against the CPU oracle, through the C-ABI (needs a B200).

Bar (BASELINE.json north_star): cluster membership and keypoint sets bit-exact; keypoint
coordinates and descriptor values within 1e-5 relative (they are bit-exact in practice: descriptor
bins are summed in PCL's order whatever the neighbourhood size); no whitelist of any kind.  The
tolerance-boundary report the north star asks for is a separate count (test_boundary_report...).
"""
import numpy as np
import pytest

from util import bits_equal, check_descriptors, rel_err, to_fe_params, DESC_RTOL

pytestmark = pytest.mark.gpu


def _params(ob, cfg):
    P = ob.launch_playback() if cfg == 1 else ob.node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    return P


@pytest.fixture(scope="module")
def nodes(ob):
    from feature_extraction_b200 import FeatureExtractionNode
    made = {}

    def get(cfg):
        if cfg not in made:
            made[cfg] = FeatureExtractionNode(to_fe_params(_params(ob, cfg)), max_points=8 << 20, max_scans=512,
                                              max_keypoints=1 << 15)
        return made[cfg]
    yield get
    for n in made.values():
        n.close()


@pytest.mark.parametrize("cfg", [1, 2, 3, 4])
def test_each_reference_function_matches_the_oracle(ob, synth, nodes, cfg):
    """Rows A-N of SURVEY.md §8(a), one C-ABI entry point per reference member function."""
    P = _params(ob, cfg)
    nd = nodes(cfg)
    pts, offs, rp = synth.generate(cfg, 2)
    for s in range(2):
        sc = pts[offs[s]:offs[s + 1]]
        r = ob.process_scan(P, sc, rp[s, 0], rp[s, 1], mode=0)
        # A getElevationAngles (src:147-156)
        el_o = ob.get_elevation_angles(sc)
        assert bits_equal(nd.getElevationAngles(sc), el_o)
        # B rotateCloud (src:159-167)
        nd.roll, nd.pitch = rp[s]
        assert bits_equal(nd.rotateCloud(el_o), ob.rotate_cloud(el_o, rp[s, 0], rp[s, 1]))
        assert bits_equal(nd.rotateCloud(el_o), r["cloud_full"])
        # D filterCloud (src:169-183)
        assert bits_equal(nd.filterCloud(r["cloud_full"]), r["cloud"])
        # E2 EuclideanClusterExtraction per ring (src:269-276): membership, member order, cluster order
        for ring in (3, 6, 9):
            rc = ob.select_ring(r["cloud"], ring)
            if len(rc) == 0 or len(rc) > 2900:
                continue
            co = ob.extract_clusters(rc, P.cluster_tolerance, P.cluster_min_count, P.cluster_max_count)
            cg = nd.extractClusters(rc, P.cluster_tolerance, P.cluster_min_count, P.cluster_max_count)
            assert len(co) == len(cg)
            assert all(np.array_equal(a, b) for a, b in zip(co, cg))
            # F getCylinderSegments (src:261-327)
            cen_o, cc_o = ob.get_cylinder_segments(P, rc)
            cen_g, cc_g = nd.getCylinderSegments(rc)
            assert bits_equal(cen_g, cen_o) and bits_equal(cc_g, cc_o)
        # E1+G estimateKeypoints (src:185-259)
        kp_o, kc_o, _ = ob.estimate_keypoints(P, r["cloud"])
        kp_g, kc_g = nd.estimateKeypoints(r["cloud"])
        assert bits_equal(kp_g, kp_o) and bits_equal(kc_g, kc_o)
        assert bits_equal(kp_o, r["keypoints"])
        # H-N estimateDescriptors (src:329-355)
        if len(kp_o):
            d_g = nd.estimateDescriptors(r["cloud_full"], kp_o)
            ok, bad = check_descriptors(d_g, r["descriptors"])
            assert bad == 0, (ok, bad)


@pytest.mark.parametrize("cfg,nscans", [(1, 6), (2, 48), (3, 3), (4, 4)])
def test_fused_batch_matches_the_oracle(ob, synth, nodes, cfg, nscans):
    """cloudCallback (src:83-117) in batch form, plus the ~cloud / ~keypoint_cloud outputs."""
    P = _params(ob, cfg)
    nd = nodes(cfg)
    pts, offs, rp = synth.generate(cfg, nscans, scan_index_base=100)
    nd.enableCloudOutputs(True)
    ko, kp, d = nd.processBatch(pts, offs, rp)
    co, cloud, kco, kcloud = nd.cloudOutputs(nscans)
    nd.enableCloudOutputs(False)
    ko_o, kp_o, d_o, _ = ob.process_batch(P, pts, offs, rp, mode=0, n_threads=8)
    assert np.array_equal(ko, ko_o)
    assert bits_equal(kp, kp_o)
    ok, bad = check_descriptors(d, d_o)
    assert bad == 0, (ok, bad)
    for s in range(nscans):
        r = ob.process_scan(P, pts[offs[s]:offs[s + 1]], rp[s, 0], rp[s, 1], mode=1)
        assert bits_equal(cloud[co[s]:co[s + 1]], r["cloud"])
        assert bits_equal(kcloud[kco[s]:kco[s + 1]], r["keypoint_cloud"])


def test_many_equal_size_clusters_follow_libstdcxx_sort_order(ob, nodes):
    """> 16 clusters with ties: PCL's final std::sort is not stable; the device replays it."""
    nd = nodes(2)
    rng = np.random.default_rng(11)
    for trial in range(6):
        ncl = int(rng.integers(20, 150))
        pts = []
        for c in range(ncl):
            size = int(rng.integers(1, 5))
            cx, cy = 2.0 * (c % 40), 2.0 * (c // 40)
            for k in range(size):
                pts.append((cx + 0.05 * k, cy + 0.01 * rng.normal(), 0.0, -1.0))
        pts = np.array(pts, np.float32)
        pts = pts[rng.permutation(len(pts))]
        co = ob.extract_clusters(pts, 0.65, 1, 1000)
        cg = nd.extractClusters(pts, 0.65, 1, 1000)
        assert len(co) == len(cg) == ncl
        assert all(np.array_equal(a, b) for a, b in zip(co, cg))


def test_device_resident_entry_point_equals_host_entry_point(ob, synth, nodes):
    import torch
    nd = nodes(2)
    pts, offs, rp = synth.generate(2, 16, scan_index_base=500)
    ko, kp, d = nd.processBatch(pts, offs, rp)
    dev = torch.from_numpy(pts).cuda()
    torch.cuda.synchronize()
    ko2, K, p_kp, p_d = nd.processBatchDevice(dev.data_ptr(), offs, rp)
    assert np.array_equal(ko, ko2) and K == len(kp)
    assert bits_equal(nd.download(p_kp, (K, 4)), kp)
    d2 = nd.download(p_d, (K, 1980))
    assert bits_equal(d2, d)
    # a handful of scans from the same device buffer: eager, captured, replayed (the pointer is part of the graph's key)
    for g0, g1 in ((0, 3), (3, 4), (0, 3), (0, 3), (3, 4), (3, 4), (0, 3)):
        o = offs[g0:g1 + 1] - offs[g0]
        ko3, K3, p_kp3, p_d3 = nd.processBatchDevice(dev.data_ptr() + int(offs[g0]) * 16, o, rp[g0:g1])
        a, b = int(ko[g0]), int(ko[g1])
        assert np.array_equal(ko3, ko[g0:g1 + 1] - a) and K3 == b - a
        assert bits_equal(nd.download(p_kp3, (K3, 4)), kp[a:b]) and bits_equal(nd.download(p_d3, (K3, 1980)), d[a:b])
    # 50 scans: the batch instantiations
    pts5, offs5, rp5 = synth.generate(2, 50, scan_index_base=520)
    ko5, kp5, d5 = nd.processBatch(pts5, offs5, rp5)
    dev5 = torch.from_numpy(pts5).cuda()
    ko6, K6, p_kp6, p_d6 = nd.processBatchDevice(dev5.data_ptr(), offs5, rp5)
    assert np.array_equal(ko5, ko6) and bits_equal(nd.download(p_kp6, (K6, 4)), kp5) and bits_equal(nd.download(p_d6, (K6, 1980)), d5)


def test_cpp_host_mirror_example_runs():
    """The C++ FeatureExtractionCore (reference method names) stage-by-stage == fused, on the GPU."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["make", "-s", "-C", os.path.join(root, "examples")])
    out = subprocess.run([os.path.join(root, "examples", "core_example")], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "identical" in out.stdout and "1 keypoints" in out.stdout


@pytest.mark.parametrize("stride,offs", [(12, (0, 4, 8)), (16, (0, 4, 8)), (32, (0, 4, 8)), (22, (0, 4, 8)), (32, (4, 12, 20)), (19, (1, 6, 11))])
def test_record_layouts_decode_on_device(ob, synth, nodes, stride, offs):
    """SURVEY.md §8(f)1: PointCloud2-style records (point_step / field offsets, incl. the 2-byte aligned
    22-byte Velodyne layout and a deliberately odd one) give the same result as fe_point_t input."""
    nd = nodes(2)
    pts, so, rp = synth.generate(2, 5, scan_index_base=900)
    ko, kp, d = nd.processBatch(pts, so, rp)
    raw = np.zeros((len(pts), stride), np.uint8)
    raw[:] = 0xAB  # junk in the unused bytes
    for k, o in enumerate(offs):
        raw[:, o:o + 4] = pts[:, k].copy().view(np.uint8).reshape(-1, 4)
    ko2, kp2, d2 = nd.processBatchLayout(raw, stride, offs[0], offs[1], offs[2], so, rp)
    assert np.array_equal(ko, ko2) and bits_equal(kp, kp2)
    from util import rel_err
    assert rel_err(d2, d).max() < 1e-5


@pytest.mark.parametrize("cfg,nscans", [(1, 3), (2, 12), (3, 6), (4, 2)])
def test_descriptors_are_bit_identical_when_summed_in_pcl_order(ob, synth, nodes, cfg, nscans):
    """Rows J/N: the contributions of a keypoint are added in ascending (d2, index) order like
    FLANN's sorted radius search delivers them, so the float sums are the oracle's bit for bit —
    also for keypoints with more contributions than the sort workspace holds (bins handled in groups)."""
    P = _params(ob, cfg)
    nd = nodes(cfg)
    pts, offs, rp = synth.generate(cfg, nscans, scan_index_base=300)
    ko, kp, d = nd.processBatch(pts, offs, rp)
    exact = total = 0
    for s in range(nscans):
        r = ob.process_scan(P, pts[offs[s]:offs[s + 1]], rp[s, 0], rp[s, 1], mode=0)
        dg = d[ko[s]:ko[s + 1]]
        assert bits_equal(kp[ko[s]:ko[s + 1]], r["keypoints"])
        for i in range(len(dg)):
            total += 1
            exact += int(bits_equal(dg[i], r["descriptors"][i]))
    assert total > 0 and exact == total, (exact, total)


def test_in_process_multi_gpu_sharding_equals_single_context(ob, synth, nodes):
    """fe_multi_*: every visible GPU (at least one) gets a contiguous scan range; the gathered CSR result
    equals the single-context result."""
    import torch
    from feature_extraction_b200 import MultiGpuExtractor
    nd = nodes(2)
    pts, offs, rp = synth.generate(2, 23, scan_index_base=1200)
    ko, kp, d = nd.processBatch(pts, offs, rp)
    for devs in ([0], list(range(torch.cuda.device_count())), [0, 0, 0]):
        m = MultiGpuExtractor(devs, to_fe_params(_params(ob, 2)), max_points=4 << 20, max_scans=64, max_keypoints=4096)
        ko2, kp2, d2 = m.processBatch(pts, offs, rp)
        m.close()
        assert np.array_equal(ko, ko2) and bits_equal(kp, kp2) and bits_equal(d, d2)


def test_record_output_equals_concatenate_fields_on_the_host(ob, synth, nodes):
    """SURVEY.md §8(f)1, output side: with fe_enable_record_output the device emits the 7,984-byte
    pcl::PointDescriptor records (feature_extraction_node.h:35-53, concatenateFields at src:119)
    itself — host, device-resident and multi-GPU entry points; sub-batching must not matter."""
    import torch
    from feature_extraction_b200 import FeatureExtractionNode, MultiGpuExtractor, pack_point_descriptors
    from feature_extraction_b200.node import RECORD_FLOATS
    nd = nodes(2)
    pts, offs, rp = synth.generate(2, 40, scan_index_base=2300)
    pts = pts.copy()
    pts[offs[7]:offs[8], 0] -= 500.0          # a scan without keypoints in the middle
    ko, kp, d = nd.processBatch(pts, offs, rp)
    want = pack_point_descriptors(kp, d)
    assert want.shape == (len(kp), RECORD_FLOATS) and len(kp) > 40
    P = to_fe_params(_params(ob, 2))
    for max_scans in (64, 9):                 # one sub-batch / five sub-batches on two slots
        r = FeatureExtractionNode(P, max_points=1 << 20, max_scans=max_scans, max_keypoints=4096)
        r.enableRecordOutput(True)
        ko2, kp2, rec = r.processBatch(pts, offs, rp)
        assert np.array_equal(ko, ko2) and bits_equal(kp, kp2) and rec.shape == want.shape
        assert bits_equal(rec, want)
        if max_scans == 64:
            dev = torch.from_numpy(pts).cuda()
            torch.cuda.synchronize()
            ko3, K, p_kp, p_rec = r.processBatchDevice(dev.data_ptr(), offs, rp)
            assert K == len(kp) and bits_equal(r.download(p_rec, (K, RECORD_FLOATS)), want)
            r.enableRecordOutput(False)       # back to plain bins on the same context
            ko4, kp4, d4 = r.processBatch(pts, offs, rp)
            assert d4.shape == d.shape and bits_equal(d4, d)
        r.close()
    m = MultiGpuExtractor([0, 0], P, max_points=1 << 20, max_scans=64, max_keypoints=4096)
    m.enableRecordOutput(True)
    ko5, kp5, rec5 = m.processBatch(pts, offs, rp)
    m.close()
    assert np.array_equal(ko, ko5) and bits_equal(rec5, want)
    # descriptors off: no records, not an error
    P0 = to_fe_params(_params(ob, 2))
    P0.estimate_descriptors = 0
    r = FeatureExtractionNode(P0, max_points=1 << 20, max_scans=64, max_keypoints=4096)
    r.enableRecordOutput(True)
    ko6, kp6, rec6 = r.processBatch(pts, offs, rp)
    r.close()
    assert rec6 is None and bits_equal(kp6, kp)


def test_stage_timing_mode_serialises_without_changing_results(ob, synth, nodes):
    """fe_enable_stage_timing: small calls run eagerly instead of from a captured graph, every stage
    gets a CUDA-event pair; results stay bit-identical and fe_get_stage_times reports the stages."""
    import torch
    nd = nodes(2)
    pts, offs, rp = synth.generate(2, 48, scan_index_base=4100)
    ko, kp, d = nd.processBatch(pts, offs, rp)
    assert nd.stageTimes() == []                      # not collected by default
    nd.enableStageTiming(True)
    try:
        ko2, kp2, d2 = nd.processBatch(pts, offs, rp)
        names = [n for n, ms in nd.stageTimes()]
        dev = torch.from_numpy(pts).cuda()
        torch.cuda.synchronize()
        ko3, K, p_kp, p_d = nd.processBatchDevice(dev.data_ptr(), offs, rp)
        names_dev = [n for n, ms in nd.stageTimes()]
        d3 = nd.download(p_d, (K, 1980))
    finally:
        nd.enableStageTiming(False)
    assert np.array_equal(ko, ko2) and bits_equal(kp, kp2) and bits_equal(d, d2)
    assert np.array_equal(ko, ko3) and bits_equal(d, d3)
    for want in ("K1 level+crop+ring", "K2 ring clusters", "K3 merge keypoints", "K4a surface grid", "K4b mark neighbours",
                 "K4c density", "K4d shape context"):
        assert want in names and want in names_dev


@pytest.mark.parametrize("cfg,nscans", [(1, 6), (2, 64), (3, 4), (4, 6)])
def test_run_based_and_grid_based_ring_clustering_agree(ob, synth, nodes, cfg, nscans):
    """Row E2/F two ways: the run-based K2 (rings in firing order cut into runs, links between runs) and
    the grid-based kernels it falls back to (cell grid + union-find) must give the oracle's keypoints and
    keypoint_cloud bit for bit — also on rings whose entries arrive in arbitrary order, where every entry
    is a run of its own and scans with more than 256 runs in a ring take the fallback."""
    P = _params(ob, cfg)
    nd = nodes(cfg)
    pts, offs, rp = synth.generate(cfg, nscans, scan_index_base=7700)
    ko_o, kp_o, _, _ = ob.process_batch(P, pts, offs, rp, mode=1, n_threads=8, want_desc=False)
    nd.enableCloudOutputs(True)
    res = {}
    for grid in (False, True):
        nd.forceGridClustering(grid)
        ko, kp, d = nd.processBatch(pts, offs, rp)
        res[grid] = (ko, kp, d) + nd.cloudOutputs(nscans)
    nd.forceGridClustering(False)
    nd.enableCloudOutputs(False)
    for grid in (False, True):
        assert np.array_equal(res[grid][0], ko_o) and bits_equal(res[grid][1], kp_o), grid
    assert np.array_equal(res[False][5], res[True][5]) and bits_equal(res[False][6], res[True][6])  # ~keypoint_cloud
    # the same scans with every scan's points shuffled: same clusters, other order of discovery
    rng = np.random.default_rng(3)
    n2 = min(nscans, 3)
    sh = pts[: offs[n2]].copy()
    for s in range(n2):
        sh[offs[s]:offs[s + 1]] = sh[offs[s]:offs[s + 1]][rng.permutation(int(offs[s + 1] - offs[s]))]
    ko_o, kp_o, _, _ = ob.process_batch(P, sh, offs[: n2 + 1], rp[:n2], mode=1, n_threads=8, want_desc=False)
    ko, kp, d = nd.processBatch(sh, offs[: n2 + 1], rp[:n2])
    assert np.array_equal(ko, ko_o) and bits_equal(kp, kp_o)


def test_cloud_outputs_across_sub_batches_and_shards(ob, synth):
    """~cloud (src:137-139) and ~keypoint_cloud (src:133-135) of a call that the library cuts into several
    sub-batches (two slots, device-side gather into pinned memory), and of the in-process multi-GPU form,
    equal the oracle's per-scan clouds bit for bit."""
    from feature_extraction_b200 import FeatureExtractionNode, MultiGpuExtractor
    P = ob.node_default()
    pts, offs, rp = synth.generate(2, 37, scan_index_base=9100)
    pts = pts.copy()
    pts[offs[11]:offs[12], 0] -= 500.0    # a scan that is cropped away entirely, in the middle
    want = [ob.process_scan(P, pts[offs[s]:offs[s + 1]], rp[s, 0], rp[s, 1], mode=1) for s in range(37)]
    nd = FeatureExtractionNode(to_fe_params(P), max_points=1 << 20, max_scans=8, max_keypoints=4096)   # 5 sub-batches
    nd.enableCloudOutputs(True)
    for rep in range(2):                  # the second call reuses (and may regrow) the pinned result buffers
        ko, kp, d = nd.processBatch(pts, offs, rp)
        co, cloud, kco, kcloud = nd.cloudOutputs(37)
        for s in range(37):
            assert bits_equal(cloud[co[s]:co[s + 1]], want[s]["cloud"]), s
            assert bits_equal(kcloud[kco[s]:kco[s + 1]], want[s]["keypoint_cloud"]), s
            assert bits_equal(kp[ko[s]:ko[s + 1]], want[s]["keypoints"]), s
    nd.close()
    m = MultiGpuExtractor([0, 0, 0], to_fe_params(P), max_points=1 << 20, max_scans=5, max_keypoints=4096)
    m.enableCloudOutputs(True)
    ko, kp, d = m.processBatch(pts, offs, rp)
    co, cloud, kco, kcloud = m.cloudOutputs(37)
    m.close()
    for s in range(37):
        assert bits_equal(cloud[co[s]:co[s + 1]], want[s]["cloud"]), s
        assert bits_equal(kcloud[kco[s]:kco[s + 1]], want[s]["keypoint_cloud"]), s


def test_single_scan_calls_replay_a_captured_graph(ob, synth):
    """The reference's deployment is one scan per callback (src:72, ros::spin): small sub-batches are captured
    into a CUDA graph per shape and replayed.  Replays, eager launches and the oracle agree bit for bit; a
    parameter change or another output mode invalidates the captured graphs."""
    from feature_extraction_b200 import FeatureExtractionNode
    P = ob.launch_playback()
    nd = FeatureExtractionNode(to_fe_params(P), max_points=1 << 18, max_scans=4, max_keypoints=1024)
    pts, offs, rp = synth.generate(1, 6, scan_index_base=9400)
    want = [ob.process_scan(P, pts[offs[s]:offs[s + 1]], rp[s, 0], rp[s, 1], mode=1) for s in range(6)]
    one = np.array([0, 0], np.int64)
    for rep in range(3):
        for s in range(6):
            sc = pts[offs[s]:offs[s + 1]]
            one[1] = len(sc)
            ko, kp, d = nd.processBatch(sc, one, rp[s:s + 1])
            assert bits_equal(kp, want[s]["keypoints"]) and bits_equal(d, want[s]["descriptors"]), (rep, s)
    replays = nd.enableGraphs(True)
    assert replays >= 6          # scans of equal chunk count share a graph from their second sighting on
    nd.enableGraphs(False)       # eager launches give the same
    sc = pts[offs[2]:offs[3]]
    one[1] = len(sc)
    ko, kp, d = nd.processBatch(sc, one, rp[2:3])
    assert bits_equal(kp, want[2]["keypoints"]) and bits_equal(d, want[2]["descriptors"])
    assert nd.enableGraphs(True) == replays
    # new parameters: the old graphs must not be replayed
    P2 = ob.node_default()
    nd.set_params(to_fe_params(P2))
    w2 = ob.process_scan(P2, sc, rp[2, 0], rp[2, 1], mode=1)
    for rep in range(3):
        ko, kp, d = nd.processBatch(sc, one, rp[2:3])
        assert bits_equal(kp, w2["keypoints"]) and bits_equal(d, w2["descriptors"])
    nd.enableCloudOutputs(True)
    for rep in range(3):
        ko, kp, d = nd.processBatch(sc, one, rp[2:3])
        co, cloud, kco, kcloud = nd.cloudOutputs(1)
        assert bits_equal(kp, w2["keypoints"]) and bits_equal(cloud, w2["cloud"]) and bits_equal(kcloud, w2["keypoint_cloud"])
    # a scan without keypoints and an empty scan through the same context
    far = sc.copy()
    far[:, 0] -= 500.0
    for rep in range(3):
        ko, kp, d = nd.processBatch(far, one, rp[2:3])
        assert ko[-1] == 0
    ko, kp, d = nd.processBatch(np.zeros((0, 4), np.float32), np.zeros(2, np.int64), rp[2:3])
    assert ko[-1] == 0
    nd.close()


@pytest.mark.parametrize("cfg,nscans", [(1, 20), (2, 24), (3, 18), (4, 20)])
def test_small_sub_batch_kernels_agree_with_the_batch_kernels(ob, synth, nodes, cfg, nscans):
    """Calls of at most 16 scans (the reference's one scan per callback) run K2 with a warp per ring and K4d with a
    block per keypoint; larger calls run the throughput instantiations.  Both must give the oracle's bits."""
    P = _params(ob, cfg)
    nd = nodes(cfg)
    pts, offs, rp = synth.generate(cfg, nscans, scan_index_base=12300)
    ko_b, kp_b, d_b = nd.processBatch(pts, offs, rp)          # > 16 scans: batch kernels
    ko_o, kp_o, d_o, _ = ob.process_batch(P, pts, offs, rp, mode=1, n_threads=4)
    assert np.array_equal(ko_b, ko_o) and bits_equal(kp_b, kp_o) and bits_equal(d_b, d_o)
    for g0 in range(0, nscans, 5):                              # 5 scans per call: small-batch kernels
        g1 = min(g0 + 5, nscans)
        o = offs[g0:g1 + 1] - offs[g0]
        ko, kp, d = nd.processBatch(pts[offs[g0]:offs[g1]], o, rp[g0:g1])
        a, b = ko_o[g0], ko_o[g1]
        assert np.array_equal(ko, ko_o[g0:g1 + 1] - a), (cfg, g0)
        assert bits_equal(kp, kp_o[a:b]) and bits_equal(d, d_o[a:b]), (cfg, g0)


def test_lean_chain_runs_a_deferring_scan_again_with_the_fallback_kernels(ob, synth):
    """Small sub-batches run only the first instantiation of every stage; a scan one of them defers (here: a
    shuffled cloud, every ring entry a run of its own) is run again with the whole chain, and the lean chain stays
    off for a while.  Results are the oracle's either way."""
    from feature_extraction_b200 import FeatureExtractionNode
    P = ob.node_default()
    nd = FeatureExtractionNode(to_fe_params(P), max_points=1 << 18, max_scans=4, max_keypoints=2048)
    pts, offs, rp = synth.generate(2, 3, scan_index_base=31000)
    one = np.array([0, 0], np.int64)
    rng = np.random.default_rng(5)
    sc0 = pts[offs[0]:offs[1]]
    dense, doffs, _ = synth.generate(3, 1, scan_index_base=31100)   # ~1,200 entries per ring: far beyond RW2 runs
    shuf = dense[rng.permutation(len(dense))]
    w_shuf = ob.process_scan(P, shuf, rp[0, 0], rp[0, 1], mode=1)
    w0 = ob.process_scan(P, sc0, rp[0, 0], rp[0, 1], mode=1)
    for rep in range(3):                   # eager, capture, replay of the lean chain
        one[1] = len(sc0)
        ko, kp, d = nd.processBatch(sc0, one, rp[0:1])
        assert bits_equal(kp, w0["keypoints"]) and bits_equal(d, w0["descriptors"])
    assert nd.leanReruns() == 0
    r0 = nd.leanReruns()
    for rep in range(3):
        one[1] = len(shuf)
        ko, kp, d = nd.processBatch(shuf, one, rp[0:1])
        assert bits_equal(kp, w_shuf["keypoints"]) and bits_equal(d, w_shuf["descriptors"]), rep
    assert nd.leanReruns() == r0 + 1      # the first one was run again; after that the whole chain runs at once
    for rep in range(3):                   # and ordered scans are still right while the lean chain is held off
        one[1] = len(sc0)
        ko, kp, d = nd.processBatch(sc0, one, rp[0:1])
        assert bits_equal(kp, w0["keypoints"]) and bits_equal(d, w0["descriptors"])
    nd.close()


def test_bench_dump_outputs_are_the_oracles_results(ob, synth, tmp_path):
    """bench.py --dump-outputs: the device-resident results of the last timed step of the main configuration,
    float32/float64 .npy files, equal to the oracle's on the batch the bench generates (rank 0: scans 0..B-1)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--config", "4", "--scans", "6", "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    got = {n: np.load(tmp_path / (n + ".npy")) for n in ("keypoint_offsets", "keypoints", "descriptors", "descriptor_rows")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    pts, offs, rp = synth.generate(4, 6)
    ko_o, kp_o, d_o, _ = ob.process_batch(_params(ob, 4), pts, offs, rp, mode=1, n_threads=4)
    assert len(kp_o) > 0 and np.array_equal(got["keypoint_offsets"], ko_o) and bits_equal(got["keypoints"], kp_o)
    assert np.array_equal(got["descriptor_rows"], np.arange(len(kp_o))) and bits_equal(got["descriptors"], d_o)
