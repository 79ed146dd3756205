"""Host-side logic of the product library that needs no GPU: the C-ABI loads and exports every
symbol include/fe_b200.h declares, host helpers agree with the oracle, and the library fails
loudly (no CPU fallback) when no device is present."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from feature_extraction_b200 import _native
    lib = _native.lib()
    header = open(os.path.join(ROOT, "include", "fe_b200.h")).read()
    declared = set(re.findall(r"\b(fe_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)
    for sym in declared:
        assert getattr(lib, sym) is not None
    assert b"sm_100a" in lib.fe_version()


def test_struct_layouts_match_the_header():
    from feature_extraction_b200 import _native
    assert C.sizeof(_native.Params) == 6 * 8 + 8 + 4 + 4 + 8 + 4 + 4 + 8
    assert C.sizeof(_native.Limits) == 32
    assert C.sizeof(_native.BatchResult) == 56


def test_presets_match_the_reference_defaults(ob):
    from feature_extraction_b200 import node_default, launch_playback
    for mine, theirs in ((node_default(), ob.node_default()), (launch_playback(), ob.launch_playback())):
        for f, _ in mine._fields_:
            assert getattr(mine, f) == getattr(theirs, f), f


def test_rotation_matrix_host_helper_matches_oracle(ob):
    from feature_extraction_b200 import rotation_matrix
    rng = np.random.default_rng(0)
    for _ in range(200):
        r, p = rng.uniform(-3.5, 3.5, 2)
        assert np.array_equal(rotation_matrix(r, p).view(np.uint32), ob.rotation_matrix(r, p).view(np.uint32))
    assert np.array_equal(rotation_matrix(0.0, 0.0), np.eye(3, dtype=np.float32))


def test_sort_replay_matches_libstdcxx_std_sort(ob):
    from feature_extraction_b200.node import debug_sort_replay
    rng = np.random.default_rng(5)
    for t in range(1500):
        n = int(rng.integers(1, 400))
        hi = int(rng.integers(2, 60))
        sizes = rng.integers(1, hi, n).astype(np.int32)
        assert np.array_equal(debug_sort_replay(sizes), ob.std_sort_cluster_order(sizes))
    # structured inputs: sorted, reversed, organ pipe, constant, few distinct values, large n
    for n in (17, 33, 100, 1000, 5000):
        base = np.arange(n, dtype=np.int32)
        for sizes in (base, base[::-1].copy(), np.minimum(base, n - base), np.ones(n, np.int32), base % 3, base % 2):
            sizes = np.ascontiguousarray(sizes, np.int32)
            assert np.array_equal(debug_sort_replay(sizes), ob.std_sort_cluster_order(sizes))


def test_sort_replay_heapsort_fallback_path(ob):
    """Drive std::sort past its depth limit (median-of-3 killer) so the heap-sort branch runs."""
    from feature_extraction_b200.node import debug_sort_replay
    for n in (64, 256, 1024, 4096):
        # Musser's median-of-3 killer sequence (on the reversed view the sort sees)
        k = n // 2
        a = np.zeros(n, np.int32)
        for i in range(1, k + 1):
            if i % 2 == 1:
                a[i - 1] = i
                a[i] = k + i
            a[k + i - 1] = 2 * i
        sizes = a[::-1].copy()
        assert np.array_equal(debug_sort_replay(sizes), ob.std_sort_cluster_order(sizes))


def test_pack_point_descriptors_layout():
    from feature_extraction_b200 import pack_point_descriptors
    kp = np.array([[1, 2, 3, 4], [5, 6, 7, 8]], np.float32)
    d = np.arange(2 * 1980, dtype=np.float32).reshape(2, 1980)
    rec = pack_point_descriptors(kp, d)
    assert rec.shape == (2, 1996) and rec.nbytes == 2 * 7984
    assert list(rec[1, :5]) == [5, 6, 7, 0, 8]
    assert np.array_equal(rec[1, 5:1985], d[1])
    assert np.all(rec[:, 1985:] == 0)


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from feature_extraction_b200 import FeatureExtractionNode, FeatureExtractionError, _native
    with pytest.raises(FeatureExtractionError) as e:
        FeatureExtractionNode()
    assert e.value.status == _native.FE_ERR_NO_DEVICE
    assert _native.lib().fe_device_count() == 0


def test_product_package_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "feature_extraction_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", "Makefile")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "oracle_binding" not in txt and "libfe_oracle" not in txt and "fe_oracle" not in txt, (dp, f)


def test_cpp_host_mirror_builds_against_the_c_abi():
    """include/feature_extraction_b200/feature_extraction_core.hpp + examples/core_example.cpp compile
    and link with nothing but the C-ABI (no CUDA, PCL or ROS headers)."""
    import subprocess
    subprocess.check_call(["make", "-s", "-B", "-C", os.path.join(ROOT, "examples")])
    assert os.path.exists(os.path.join(ROOT, "examples", "core_example"))


def test_imu_to_roll_pitch_matches_oracle_and_known_cases(ob):
    """imuCallback (src:57-70): tf getRPY, roll = tmproll - pi; zeros when cloud_leveling is false."""
    from feature_extraction_b200 import imu_to_roll_pitch
    r, p = imu_to_roll_pitch([0, 0, 0, 1])
    assert r == -np.pi and p == 0.0
    # a sensor mounted upside down (roll = pi) is what the "- pi" is there for
    r, p = imu_to_roll_pitch([1, 0, 0, 0])
    assert abs(r) < 1e-12 and abs(p) < 1e-12
    assert imu_to_roll_pitch([0.3, 0.1, -0.2, 0.9], cloud_leveling=False) == (0.0, 0.0)
    rng = np.random.default_rng(9)
    for _ in range(500):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        assert imu_to_roll_pitch(q) == ob.imu_to_roll_pitch(q)
    # pitch = 30 deg about y, then check against the closed form
    a = np.deg2rad(30.0)
    r, p = imu_to_roll_pitch([0, np.sin(a / 2), 0, np.cos(a / 2)])
    assert abs(p - a) < 1e-12 and abs(r + np.pi) < 1e-12


def test_null_and_invalid_arguments_are_status_codes_not_crashes():
    """No exception or crash crosses the C-ABI: bad arguments come back as FE_ERR_INVALID."""
    from feature_extraction_b200 import _native as N
    L = N.lib()
    res = N.BatchResult()
    assert L.fe_process_batch(None, None, None, None, 0, C.byref(res)) == N.FE_ERR_INVALID
    assert L.fe_process_batch_device(None, None, None, None, 0, C.byref(res)) == N.FE_ERR_INVALID
    assert L.fe_create(0, None, None, None) == N.FE_ERR_INVALID
    assert L.fe_set_params(None, None) == N.FE_ERR_INVALID
    assert L.fe_get_elevation_angles(None, None, 0) == N.FE_ERR_INVALID
    assert L.fe_filter_cloud(None, None, 0, None, 0, None) == N.FE_ERR_INVALID
    assert L.fe_estimate_descriptors(None, None, 0, None, 0, None) == N.FE_ERR_INVALID
    assert L.fe_rotation_matrix(0.0, 0.0, None) == N.FE_ERR_INVALID
    assert L.fe_pack_point_descriptors(None, None, 1, None) == N.FE_ERR_INVALID
    assert L.fe_pack_point_descriptors(None, None, 0, None) == N.FE_OK
    L.fe_destroy(None)  # no-op
    assert L.fe_last_error(None) == b"null context"
    lay = N.PointLayout(8, 0, 4, 8)
    assert L.fe_process_batch_layout(None, None, C.byref(lay), None, None, 0, C.byref(res)) == N.FE_ERR_INVALID


def test_multi_gpu_helper_rejects_bad_arguments():
    from feature_extraction_b200 import _native as N, node_default
    L = N.lib()
    m = C.c_void_p()
    P = node_default()
    assert L.fe_multi_create(None, 0, C.byref(P), None, C.byref(m)) == N.FE_ERR_INVALID
    res = N.BatchResult()
    assert L.fe_multi_process_batch(None, None, None, None, 0, C.byref(res)) == N.FE_ERR_INVALID
    L.fe_multi_destroy(None)
    assert L.fe_multi_last_error(None) == b"null context"


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): exactly one JSON line on
    stdout with the contract's keys, no GPU needed."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample", "24"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "scans/sec" and d["unit"] == "scans/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_bench_rejects_zero_steps_and_dumps_outside_the_device_path():
    import subprocess
    import sys
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"], ["--config", "5", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and "error:" in out.stderr, (extra, out.stderr[-2000:])


def test_bench_dump_outputs_samples_descriptor_rows_with_a_fixed_seed(tmp_path):
    """bench.py's dump_outputs on more keypoints than DUMP_DESCRIPTOR_ROWS: float32/float64 files within
    DUMP_MAX_BYTES, every keypoint, and the same seeded sample of descriptor rows on every call."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class Node:  # FeatureExtractionNode.download over host arrays keyed by "device pointer"
        def __init__(self, arrays):
            self.arrays = arrays

        def download(self, ptr, shape, dtype=np.float32):
            return self.arrays[ptr].reshape(shape).copy()

    rng = np.random.default_rng(5)
    K = bench.DUMP_DESCRIPTOR_ROWS + 1000
    kp = rng.standard_normal((K, 4)).astype(np.float32)
    desc = rng.standard_normal((K, 1980)).astype(np.float32)
    ko = np.array([0, 7, 7, K], np.int64)
    got = []
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), Node({1: kp, 2: desc}), ko, K, 1, 2)
        got.append({n: np.load(tmp_path / run / (n + ".npy")) for n in ("keypoint_offsets", "keypoints", "descriptors", "descriptor_rows")})
    a, b = got
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_MAX_BYTES
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert np.array_equal(a["keypoint_offsets"], ko) and np.array_equal(a["keypoints"], kp)
    rows = a["descriptor_rows"].astype(np.int64)
    assert len(rows) == bench.DUMP_DESCRIPTOR_ROWS and np.all(np.diff(rows) > 0) and rows[-1] < K
    assert np.array_equal(a["descriptors"], desc[rows])
    assert all(np.array_equal(a[n], b[n]) for n in a)


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """The boundary is a C ABI: include/fe_b200.h must compile as C99 and a C program must link
    against the library (no C++ types or name mangling in the exported interface)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "c_abi.c"
    src.write_text('#include <stdio.h>\n#include "fe_b200.h"\n'
                   'int main(void) { fe_params_t p; fe_params_node_default(&p);\n'
                   '  printf("%s %d %d\\n", fe_version(), (int)p.cluster_min_count, fe_device_count());\n'
                   '  return fe_create(0, &p, NULL, NULL) == FE_OK; }\n')
    exe = tmp_path / "c_abi"
    libdir = os.path.join(root, "feature_extraction_b200", "csrc")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"),
                           str(src), "-o", str(exe), "-L", libdir, "-lfe_b200", "-Wl,-rpath," + libdir])
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and " 5 " in out.stdout, out.stdout + out.stderr
