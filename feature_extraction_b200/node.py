"""Host-side mirror of the reference's FeatureExtractionNode for the per-scan path.

Same member-function names, argument meaning and early-return behaviour as
src/feature_extraction_node.cpp:147-355 of GAVLab/feature_extraction; every method forwards to
one C-ABI entry point of libfe_b200.so (include/fe_b200.h), which runs sm_100a kernels.  Clouds are
(N,4) float32 arrays {x, y, z, intensity}.  ROS / PointCloud2 I/O is not part of this package.
"""
import ctypes as C

import numpy as np

from . import _native as N

DESC_LEN = N.DESC_LEN
RECORD_FLOATS = N.RECORD_FLOATS


class FeatureExtractionError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("fe_b200 status %d: %s" % (status, message))
        self.status = status


def node_default():
    """Constructor defaults (reference src:9-34)."""
    p = N.Params()
    N.lib().fe_params_node_default(C.byref(p))
    return p


def launch_playback():
    """launch/keypoint_playback.launch:17-33 preset."""
    p = N.Params()
    N.lib().fe_params_launch_playback(C.byref(p))
    return p


def _cloud(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] != 4:
        a = a.reshape(-1, 4)
    return a


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _batch_args(n_records, scan_offsets, roll_pitch):
    """Validate a CSR batch before raw pointers cross the C-ABI (the library trusts its caller's sizes)."""
    offs = np.ascontiguousarray(scan_offsets, np.int64).reshape(-1)
    if len(offs) < 1:
        raise ValueError("scan_offsets needs n_scans + 1 entries")
    B = len(offs) - 1
    rp = np.ascontiguousarray(roll_pitch, np.float64).reshape(-1)
    if len(rp) != 2 * B:
        raise ValueError("roll_pitch needs 2 values per scan: got %d for %d scans" % (len(rp), B))
    if offs[0] < 0 or np.any(np.diff(offs) < 0):
        raise ValueError("scan_offsets must start at >= 0 and be non-decreasing")
    if n_records is not None and offs[-1] > n_records:
        raise ValueError("scan_offsets[-1] = %d exceeds the %d records passed" % (offs[-1], n_records))
    return offs, rp, B


def _descriptor_rows(a):
    """(K, 1980) bins or (K, 1996) records -> (array kept alive, row stride in floats, pointer to the first bin)."""
    a = np.ascontiguousarray(a, np.float32)
    if a.ndim != 2 or a.shape[1] not in (DESC_LEN, RECORD_FLOATS):
        raise ValueError("descriptors must be (K, %d) bins or (K, %d) records, got %s" % (DESC_LEN, RECORD_FLOATS, a.shape))
    first = 5 if a.shape[1] == RECORD_FLOATS else 0  # x, y, z, pad, intensity, then the bins
    return a, a.shape[1], C.c_void_p(a.ctypes.data + 4 * first if len(a) else None)


def _match_offsets(query_offsets, ref_offsets, n_query, n_ref):
    """Validate the groups of a match call before raw pointers cross the C-ABI; None for both = one group of all rows."""
    if query_offsets is None and ref_offsets is None and n_query is not None:
        query_offsets, ref_offsets = [0, n_query], [0, n_ref]
    if query_offsets is None or ref_offsets is None:
        raise ValueError("query_offsets and ref_offsets go together")
    qo = np.ascontiguousarray(query_offsets, np.int64).reshape(-1)
    ro = np.ascontiguousarray(ref_offsets, np.int64).reshape(-1)
    if len(qo) < 1 or len(qo) != len(ro):
        raise ValueError("query_offsets and ref_offsets need the same n_groups + 1 entries (got %d and %d)" % (len(qo), len(ro)))
    for name, o, n in (("query_offsets", qo, n_query), ("ref_offsets", ro, n_ref)):
        if o[0] < 0 or np.any(np.diff(o) < 0):
            raise ValueError("%s must start at >= 0 and be non-decreasing" % name)
        if n is not None and o[-1] > n:
            raise ValueError("%s[-1] = %d exceeds the %d rows passed" % (name, o[-1], n))
    return qo, ro, len(qo) - 1


def _unpack_match(res):
    n = int(res.n_queries)
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int32), np.zeros(0, np.float32), np.zeros(0, np.float32)
    return (np.ctypeslib.as_array(res.best, shape=(n,)).copy(), np.ctypeslib.as_array(res.shift, shape=(n,)).copy(),
            np.ctypeslib.as_array(res.dist2, shape=(n,)).copy(), np.ctypeslib.as_array(res.second_dist2, shape=(n,)).copy())


def register_params_default(**overrides):
    """fe_register_params_default, with any field overridden by keyword."""
    p = N.RegisterParams()
    N.lib().fe_register_params_default(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise ValueError("fe_register_params_t has no field %r" % k)
        setattr(p, k, v)
    return p


def _keypoint_rows(a):
    a = np.ascontiguousarray(a, np.float32)
    if a.ndim != 2 or a.shape[1] != 4:
        raise ValueError("keypoints must be (K, 4) float32 {x, y, z, elevation}, got %s" % (a.shape,))
    return a


def _unpack_register(res):
    G, n = int(res.n_groups), int(res.n_queries)

    def arr(p, shape, dtype):
        if int(np.prod(shape)) == 0:
            return np.zeros(shape, dtype)
        return np.ctypeslib.as_array(p, shape=shape).copy()
    return {"pose": arr(res.pose, (G, 4), np.float64), "rms": arr(res.rms, (G,), np.float64),
            "n_inliers": arr(res.n_inliers, (G,), np.int32), "n_hypotheses": arr(res.n_hypotheses, (G,), np.int32),
            "status": arr(res.status, (G,), np.int32), "assoc": arr(res.assoc, (n,), np.int64)}


class PinnedBuffer:
    """Page-locked host memory from fe_host_alloc, exposed as a numpy array."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(s) for s in shape)
        self.dtype = np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self._ptr = N.lib().fe_host_alloc(C.c_int64(max(nbytes, 1)))
        if not self._ptr:
            raise MemoryError("fe_host_alloc(%d) failed" % nbytes)
        buf = (C.c_char * max(nbytes, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self._ptr:
            self.array = None
            N.lib().fe_host_free(C.c_void_p(self._ptr))
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class FeatureExtractionNode:
    """The per-scan pipeline of the reference node, on one B200.

    Members mirror feature_extraction_node.h:115-127 (through `params`); `roll`/`pitch` are the
    state imuCallback leaves (src:63-65).  Not thread-safe, like the reference (ros::spin).
    """

    record_output = False  # see enableRecordOutput


    def __init__(self, params=None, device=0, max_points=0, max_scans=0, max_keypoints=0, max_ring_clusters=0):
        self._ctx = C.c_void_p()
        self.params = (params or node_default()).copy()
        self.roll = 0.0
        self.pitch = 0.0
        lim = N.Limits(max_points, max_scans, max_keypoints, max_ring_clusters)
        st = N.lib().fe_create(C.c_int(device), C.byref(self.params), C.byref(lim), C.byref(self._ctx))
        if st != N.FE_OK:
            self._ctx = C.c_void_p()
            msg = {N.FE_ERR_NO_DEVICE: "no usable sm_100 CUDA device (there is no CPU fallback)"}.get(st, "fe_create failed")
            raise FeatureExtractionError(st, msg)

    # -- lifecycle ---------------------------------------------------------------------------
    def close(self):
        if self._ctx:
            N.lib().fe_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st):
        if st != N.FE_OK:
            raise FeatureExtractionError(st, (N.lib().fe_last_error(self._ctx) or b"").decode())

    def set_params(self, params):
        self.params = params.copy()
        self._check(N.lib().fe_set_params(self._ctx, C.byref(self.params)))

    # -- one method per reference member function ------------------------------------------------
    def getElevationAngles(self, cloud):
        """src:147-156.  Returns the cloud with intensity = elevation angle (deg)."""
        c = _cloud(cloud).copy()
        self._check(N.lib().fe_get_elevation_angles(self._ctx, _ptr(c), len(c)))
        return c

    def rotateCloud(self, cloud):
        """src:159-167, with this node's roll/pitch."""
        c = _cloud(cloud).copy()
        self._check(N.lib().fe_rotate_cloud(self._ctx, _ptr(c), len(c), self.roll, self.pitch))
        return c

    def filterCloud(self, cloud):
        """src:169-183."""
        c = _cloud(cloud)
        out = np.empty_like(c)
        n = C.c_int64(0)
        self._check(N.lib().fe_filter_cloud(self._ctx, _ptr(c), len(c), _ptr(out), len(out), C.byref(n)))
        return out[: n.value].copy()

    def extractClusters(self, cloud, tolerance, min_size, max_size):
        """pcl::EuclideanClusterExtraction::extract as used at src:222-229 / 269-276."""
        c = _cloud(cloud)
        n = len(c)
        offs = np.zeros(n + 2, np.int32)
        idx = np.zeros(max(n, 1), np.int32)
        nc = C.c_int32(0)
        self._check(N.lib().fe_extract_clusters(self._ctx, _ptr(c), n, float(tolerance), int(min_size), int(max_size),
                                                _ptr(offs), n + 1, _ptr(idx), max(n, 1), C.byref(nc)))
        return [idx[offs[i]: offs[i + 1]].copy() for i in range(nc.value)]

    def getCylinderSegments(self, cloud):
        """src:261-327.  -> (keypoints, keypoint_cloud) of one ring's cloud."""
        c = _cloud(cloud)
        n = len(c)
        kp = np.empty((max(n, 1), 4), np.float32)
        kc = np.empty((max(n, 1), 4), np.float32)
        n1, n2 = C.c_int64(0), C.c_int64(0)
        self._check(N.lib().fe_get_cylinder_segments(self._ctx, _ptr(c), n, _ptr(kp), len(kp), C.byref(n1),
                                                     _ptr(kc), len(kc), C.byref(n2)))
        return kp[: n1.value].copy(), kc[: n2.value].copy()

    def estimateKeypoints(self, cloud):
        """src:185-259.  -> (keypoints, keypoint_cloud) of a cropped cloud."""
        c = _cloud(cloud)
        n = len(c)
        cap = max(2 * n, 1)
        kp = np.empty((cap, 4), np.float32)
        kc = np.empty((cap, 4), np.float32)
        n1, n2 = C.c_int64(0), C.c_int64(0)
        self._check(N.lib().fe_estimate_keypoints(self._ctx, _ptr(c), n, _ptr(kp), cap, C.byref(n1),
                                                  _ptr(kc), cap, C.byref(n2)))
        return kp[: n1.value].copy(), kc[: n2.value].copy()

    def debugKeypointsFull(self, cloud):
        """keypoints_full of src:205 (test hook)."""
        c = _cloud(cloud)
        cap = max(2 * len(c), 1)
        kf = np.empty((cap, 4), np.float32)
        n1 = C.c_int64(0)
        N.lib().fe_debug_keypoints_full.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
        self._check(N.lib().fe_debug_keypoints_full(self._ctx, _ptr(c), len(c), _ptr(kf), cap, C.byref(n1)))
        return kf[: n1.value].copy()

    def estimateDescriptors(self, cloud, keypoints):
        """src:329-355.  -> (K,1980) float32."""
        c = _cloud(cloud)
        kp = _cloud(keypoints)
        d = np.zeros((len(kp), DESC_LEN), np.float32)
        self._check(N.lib().fe_estimate_descriptors(self._ctx, _ptr(c), len(c), _ptr(kp), len(kp), _ptr(d)))
        return d

    def cloudCallback(self, cloud):
        """src:83-117 for one scan with this node's roll/pitch.  -> dict(keypoints, descriptors)."""
        c = _cloud(cloud)
        ko, kp, d = self.processBatch(c, np.array([0, len(c)], np.int64), np.array([[self.roll, self.pitch]]))
        return {"keypoints": kp, "descriptors": d}

    # -- batched form --------------------------------------------------------------------------
    def imuCallback(self, quat_xyzw, cloud_leveling=True):
        """src:57-70: orientation quaternion -> this node's roll/pitch state."""
        self.roll, self.pitch = imu_to_roll_pitch(quat_xyzw, cloud_leveling)

    def processBatchLayout(self, raw, stride, x_off, y_off, z_off, scan_offsets, roll_pitch, copy=True):
        """fe_process_batch_layout: `raw` is a contiguous uint8/any-dtype host buffer of records."""
        buf = np.ascontiguousarray(raw)
        lay = N.PointLayout(int(stride), int(x_off), int(y_off), int(z_off))
        offs, rp, B = _batch_args(buf.nbytes // max(int(stride), 1), scan_offsets, roll_pitch)
        res = N.BatchResult()
        self._check(N.lib().fe_process_batch_layout(self._ctx, _ptr(buf), C.byref(lay), _ptr(offs), _ptr(rp), B, C.byref(res)))
        return self._unpack(res, B, copy)

    def processBatch(self, points, scan_offsets, roll_pitch, copy=True):
        """fe_process_batch: HOST buffers in, host results out (CSR by scan).

        -> keypoint_offsets (B+1,) int64, keypoints (K,4), descriptors (K,1980) or None.
        With copy=False the arrays alias context-owned pinned memory (valid until the next call).
        """
        c = _cloud(points)
        offs, rp, B = _batch_args(len(c), scan_offsets, roll_pitch)
        res = N.BatchResult()
        self._check(N.lib().fe_process_batch(self._ctx, _ptr(c), _ptr(offs), _ptr(rp), B, C.byref(res)))
        return self._unpack(res, B, copy)

    def _unpack(self, res, B, copy):
        self.last_launches = int(res.gpu_launches)
        K = int(res.n_keypoints)
        ko = np.ctypeslib.as_array(res.keypoint_offsets, shape=(B + 1,))
        kp = np.zeros((0, 4), np.float32)
        d = None
        if K > 0:
            kp = np.ctypeslib.as_array(C.cast(res.keypoints, C.POINTER(C.c_float)), shape=(K, 4))
        if self.params.estimate_descriptors:
            d = np.zeros((0, DESC_LEN), np.float32)
            dl = RECORD_FLOATS if self.record_output else DESC_LEN
            d = np.zeros((0, dl), np.float32)
            if K > 0 and res.descriptors:
                d = np.ctypeslib.as_array(C.cast(res.descriptors, C.POINTER(C.c_float)), shape=(K, dl))
        if copy:
            return ko.copy(), kp.copy(), (d.copy() if d is not None else None)
        return ko, kp, d

    def enableRecordOutput(self, enable=True):
        """fe_enable_record_output: descriptors leave the device as (K, 1996) pcl::PointDescriptor
        records (concatenateFields, src:119) instead of (K, 1980) bins."""
        self._check(N.lib().fe_enable_record_output(self._ctx, 1 if enable else 0))
        self.record_output = bool(enable)

    def processBatchDevice(self, d_points_ptr, scan_offsets, roll_pitch):
        """fe_process_batch_device: points already in HBM (raw device pointer); results stay there.

        -> keypoint_offsets (B+1,) int64 host copy, n_keypoints, device ptr keypoints, device ptr descriptors
        """
        offs, rp, B = _batch_args(None, scan_offsets, roll_pitch)  # the device buffer's size is the caller's business
        res = N.BatchResult()
        self._check(N.lib().fe_process_batch_device(self._ctx, C.c_void_p(d_points_ptr), _ptr(offs), _ptr(rp), B, C.byref(res)))
        self.last_launches = int(res.gpu_launches)
        ko = np.ctypeslib.as_array(res.keypoint_offsets, shape=(B + 1,)).copy()
        return ko, int(res.n_keypoints), res.keypoints, res.descriptors

    def matchDescriptors(self, query, ref, query_offsets=None, ref_offsets=None):
        """fe_match_descriptors: for every query row, the reference row and azimuth shift of the smallest
        12-shift distance within its group (include/fe_b200.h).  `query` / `ref` are host arrays of (K, 1980) bins
        or (K, 1996) pcl::PointDescriptor records; no offsets = one group of all rows.
        -> best (n,) int64 (absolute reference row, -1 = none), shift (n,) int32, dist2 (n,), second_dist2 (n,) float32
        """
        q, qs, qp = _descriptor_rows(query)
        r, rs, rp = _descriptor_rows(ref)
        qo, ro, G = _match_offsets(query_offsets, ref_offsets, len(q), len(r))
        res = N.MatchResult()
        self._check(N.lib().fe_match_descriptors(self._ctx, qp, qs, _ptr(qo), rp, rs, _ptr(ro), G, C.byref(res)))
        return _unpack_match(res)

    def matchDescriptorsDevice(self, q_ptr, q_stride, q_offsets, r_ptr, r_stride, r_offsets):
        """fe_match_descriptors_device: rows already in HBM (raw device pointers, e.g. the descriptors
        processBatchDevice returns; a record pointer must point at its first bin, record base + 5 floats), queued on the
        context's stream behind the batch call.  Same results as matchDescriptors."""
        for st in (q_stride, r_stride):
            if int(st) < DESC_LEN:
                raise ValueError("a row stride must be at least %d floats, got %d" % (DESC_LEN, int(st)))
        qo, ro, G = _match_offsets(q_offsets, r_offsets, None, None)  # the device buffers' sizes are the caller's business
        if (qo[-1] > qo[0] and not q_ptr) or (ro[-1] > ro[0] and not r_ptr):
            raise ValueError("a device pointer is NULL while its side has rows")
        res = N.MatchResult()
        self._check(N.lib().fe_match_descriptors_device(self._ctx, C.c_void_p(q_ptr), int(q_stride), _ptr(qo), C.c_void_p(r_ptr),
                                                        int(r_stride), _ptr(ro), G, C.byref(res)))
        return _unpack_match(res)

    def matchDeviceBest(self):
        """fe_match_device_best: device address of the last match call's `best` (int64 per query row), for
        registerMatchesDevice."""
        p = C.c_void_p()
        self._check(N.lib().fe_match_device_best(self._ctx, C.byref(p)))
        return p.value

    def registerMatches(self, query_kp, ref_kp, best, query_offsets, ref_offsets, params=None):
        """fe_register_matches: the planar motion of every group from its matched keypoints (include/fe_b200.h,
        "registration").  Keypoints are (K, 4) host arrays addressed by absolute row; `best` as matchDescriptors returns
        it for the same offsets.  -> dict of pose (G, 4) float64 {c, s, tx, ty} mapping query xy into the reference
        frame, rms (G,), n_inliers, n_hypotheses, status (G,) int32 (0 no hypothesis, 1 too few inliers, 2 registered),
        assoc (n,) int64 (the reference row each query row is an inlier of, -1 = none)."""
        q = _keypoint_rows(query_kp)
        r = _keypoint_rows(ref_kp)
        b = np.ascontiguousarray(best, np.int64).reshape(-1)
        qo, ro, G = _match_offsets(query_offsets, ref_offsets, len(q), len(r))
        if len(b) != qo[-1] - qo[0]:
            raise ValueError("best needs one entry per query row: %d, got %d" % (qo[-1] - qo[0], len(b)))
        prm = params if params is not None else register_params_default()
        res = N.RegisterResult()
        self._check(N.lib().fe_register_matches(self._ctx, _ptr(q) if len(q) else None, _ptr(r) if len(r) else None,
                                                _ptr(b) if len(b) else None, _ptr(qo), _ptr(ro), G, C.byref(prm),
                                                C.byref(res)))
        return _unpack_register(res)

    def registerMatchesDevice(self, q_ptr, r_ptr, best_ptr, q_offsets, r_offsets, params=None):
        """fe_register_matches_device: keypoints (e.g. processBatchDevice's) and `best` (matchDeviceBest()) already in
        HBM, queued on the context's stream behind the batch and match calls.  Same results as registerMatches."""
        qo, ro, G = _match_offsets(q_offsets, r_offsets, None, None)  # the device buffers' sizes are the caller's business
        if (qo[-1] > qo[0] and not (q_ptr and best_ptr)) or (ro[-1] > ro[0] and not r_ptr):
            raise ValueError("a device pointer is NULL while its side has rows")
        prm = params if params is not None else register_params_default()
        res = N.RegisterResult()
        self._check(N.lib().fe_register_matches_device(self._ctx, C.c_void_p(q_ptr), C.c_void_p(r_ptr), C.c_void_p(best_ptr),
                                                       _ptr(qo), _ptr(ro), G, C.byref(prm), C.byref(res)))
        return _unpack_register(res)

    def scan_to_scan(self, ko, kp, descriptors, params=None):
        """Scan s against scan s - 1 of one batch result (processBatch's keypoint_offsets, keypoints, descriptors):
        match, then register.  -> registerMatches' dict for the B - 1 groups plus `best`; pose[s - 1] maps scan s's
        levelled xy into scan s - 1's."""
        ko = np.ascontiguousarray(ko, np.int64)
        best = self.matchDescriptors(descriptors, descriptors, ko[1:], ko[:-1])[0]
        out = self.registerMatches(kp, kp, best, ko[1:], ko[:-1], params)
        out["best"] = best
        return out

    def download(self, device_ptr, shape, dtype=np.float32):
        """Copy a device-resident result of processBatchDevice to a new host array."""
        out = np.empty(shape, dtype)
        if out.nbytes:
            self._check(N.lib().fe_download(self._ctx, _ptr(out), C.c_void_p(device_ptr), out.nbytes))
        return out

    def enableCloudOutputs(self, enable=True):
        self._check(N.lib().fe_enable_cloud_outputs(self._ctx, 1 if enable else 0))

    def cloudOutputs(self, n_scans):
        """~cloud (src:137-139) and ~keypoint_cloud (src:133-135) of the last host batch call."""
        co, kco = C.POINTER(C.c_int64)(), C.POINTER(C.c_int64)()
        cp, kcp = C.c_void_p(), C.c_void_p()
        self._check(N.lib().fe_get_cloud_outputs(self._ctx, C.byref(co), C.byref(cp), C.byref(kco), C.byref(kcp)))
        return _unpack_clouds(co, cp, kco, kcp, n_scans)

    def setAngleLibm(self, correctly_rounded=False):
        """fe_set_angle_libm: fdlibm atan2f/acosf (glibc <= 2.40, default) or correctly rounded (>= 2.41)."""
        self._check(N.lib().fe_set_angle_libm(self._ctx, 1 if correctly_rounded else 0))

    def enableBoundaryReport(self, eps_m=1e-6):
        """fe_enable_boundary_report: count, per scan, the pairs within eps_m of every radius predicate."""
        self._check(N.lib().fe_enable_boundary_report(self._ctx, float(eps_m)))

    def boundaryReport(self):
        """-> (n_scans, 4) int64: ring clustering, cross-ring merge, 3DSC support, 3DSC density."""
        p = C.POINTER(C.c_int64)()
        n = C.c_int32(0)
        self._check(N.lib().fe_get_boundary_report(self._ctx, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.zeros((0, 4), np.int64)
        return np.ctypeslib.as_array(p, shape=(n.value, 4)).copy()

    def enableBoundaryReportAll(self, eps_m=1e-6):
        """fe_enable_boundary_report_all: the four radius kinds plus the crop box, ring-window ends, cluster diameter
        gate and 3DSC radial, elevation and azimuth bin edges (kinds 4-9 of include/fe_b200.h)."""
        self._check(N.lib().fe_enable_boundary_report_all(self._ctx, float(eps_m)))

    def boundaryReportAll(self):
        """-> (n_scans, 10) int64: the counts of kinds 0-9 of the last batch call."""
        p = C.POINTER(C.c_int64)()
        n = C.c_int32(0)
        self._check(N.lib().fe_get_boundary_report_all(self._ctx, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.zeros((0, 10), np.int64)
        return np.ctypeslib.as_array(p, shape=(n.value, 10)).copy()

    def h2dProbe(self, host_array):
        """Bench hook: bare host->device copy of `host_array` through the staging buffer; -> ms (CUDA events)."""
        ms = C.c_float(0)
        self._check(N.lib().fe_debug_h2d_probe(self._ctx, _ptr(host_array), host_array.nbytes, C.byref(ms)))
        return float(ms.value)

    def enableGraphs(self, enable=True):
        """Test hook: CUDA-graph replay of small sub-batches on/off; -> graph replays so far."""
        n = C.c_int64(0)
        self._check(N.lib().fe_debug_enable_graphs(self._ctx, 1 if enable else 0, C.byref(n)))
        return int(n.value)

    def leanReruns(self):
        """Test hook: small sub-batches that were run again with the whole chain of fallback kernels."""
        n = C.c_int64(0)
        self._check(N.lib().fe_debug_lean_reruns(self._ctx, C.byref(n)))
        return int(n.value)

    def forceGridClustering(self, enable=True):
        """Test hook: K2 through the grid-based kernels only (the run-based kernel's fallback and cross-check)."""
        self._check(N.lib().fe_debug_force_grid_clustering(self._ctx, 1 if enable else 0))

    def debugLibm(self, op, a, b=None):
        """Test hook: the device's atan2f (op 0), acosf (1), atanf (2) element-wise."""
        a = np.ascontiguousarray(a, np.float32)
        b = np.ascontiguousarray(b if b is not None else a, np.float32)
        out = np.empty_like(a)
        self._check(N.lib().fe_debug_libm_f32(self._ctx, int(op), _ptr(a), _ptr(b), _ptr(out), a.size))
        return out

    def timerBegin(self):
        self._check(N.lib().fe_timer_begin(self._ctx))

    def timerEnd(self):
        ms = C.c_float(0)
        self._check(N.lib().fe_timer_end(self._ctx, C.byref(ms)))
        return float(ms.value)

    def batchStats(self):
        out = np.zeros(10, np.int64)
        self._check(N.lib().fe_get_batch_stats(self._ctx, _ptr(out)))
        keys = ("points", "surface_points", "crop_points", "ring_clusters", "keypoints", "neighbours",
                "deferred_ring_scans", "deferred_merge_scans", "deferred_surface_scans", "descriptors_unordered")
        st = dict(zip(keys, (int(v) for v in out)))
        w = np.zeros(3, np.int64)
        if N.lib().fe_debug_density_work(self._ctx, _ptr(w)) == N.FE_OK:
            st["density_tests"], st["marked_points"], st["halo_points"] = (int(v) for v in w)
            st["density_tests_per_marked_point"] = float(w[0]) / max(int(w[1]), 1)
        return st

    def enableStageTiming(self, enable=True):
        """fe_enable_stage_timing: serialise the stages and time each one (see stageTimes)."""
        self._check(N.lib().fe_enable_stage_timing(self._ctx, 1 if enable else 0))

    def stageTimes(self):
        names = (C.c_char_p * 32)()
        ms = (C.c_float * 32)()
        n = C.c_int32(0)
        self._check(N.lib().fe_get_stage_times(self._ctx, 32, names, ms, C.byref(n)))
        return [(names[i].decode(), float(ms[i])) for i in range(n.value)]


def _unpack_clouds(co, cp, kco, kcp, n_scans):
    co = np.ctypeslib.as_array(co, shape=(n_scans + 1,)).copy()
    kco = np.ctypeslib.as_array(kco, shape=(n_scans + 1,)).copy()

    def arr(p, n):
        if n == 0 or not p:
            return np.zeros((0, 4), np.float32)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(n, 4)).copy()
    return co, arr(cp, int(co[-1])), kco, arr(kcp, int(kco[-1]))


class MultiGpuExtractor:
    """fe_multi_*: scans sharded over several GPUs of one box in ONE process (a host thread and a
    context per GPU, contiguous scan ranges, host-side CSR gather; no collective)."""

    record_output = False


    def __init__(self, devices, params=None, max_points=0, max_scans=0, max_keypoints=0, max_ring_clusters=0):
        self._m = C.c_void_p()
        self.params = (params or node_default()).copy()
        dev = np.ascontiguousarray(devices, np.int32)
        lim = N.Limits(max_points, max_scans, max_keypoints, max_ring_clusters)
        st = N.lib().fe_multi_create(_ptr(dev), len(dev), C.byref(self.params), C.byref(lim), C.byref(self._m))
        if st != N.FE_OK:
            self._m = C.c_void_p()
            raise FeatureExtractionError(st, "fe_multi_create failed")

    def enableRecordOutput(self, enable=True):
        st = N.lib().fe_multi_enable_record_output(self._m, 1 if enable else 0)
        if st != N.FE_OK:
            raise FeatureExtractionError(st, "fe_multi_enable_record_output")
        self.record_output = bool(enable)

    def enableCloudOutputs(self, enable=True):
        st = N.lib().fe_multi_enable_cloud_outputs(self._m, 1 if enable else 0)
        if st != N.FE_OK:
            raise FeatureExtractionError(st, "fe_multi_enable_cloud_outputs")

    def cloudOutputs(self, n_scans):
        co, kco = C.POINTER(C.c_int64)(), C.POINTER(C.c_int64)()
        cp, kcp = C.c_void_p(), C.c_void_p()
        st = N.lib().fe_multi_get_cloud_outputs(self._m, C.byref(co), C.byref(cp), C.byref(kco), C.byref(kcp))
        if st != N.FE_OK:
            raise FeatureExtractionError(st, (N.lib().fe_multi_last_error(self._m) or b"").decode())
        return _unpack_clouds(co, cp, kco, kcp, n_scans)

    def close(self):
        if self._m:
            N.lib().fe_multi_destroy(self._m)
            self._m = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def processBatch(self, points, scan_offsets, roll_pitch, copy=True):
        c = _cloud(points)
        offs, rp, B = _batch_args(len(c), scan_offsets, roll_pitch)
        res = N.BatchResult()
        st = N.lib().fe_multi_process_batch(self._m, _ptr(c), _ptr(offs), _ptr(rp), B, C.byref(res))
        if st != N.FE_OK:
            raise FeatureExtractionError(st, (N.lib().fe_multi_last_error(self._m) or b"").decode())
        K = int(res.n_keypoints)
        ko = np.ctypeslib.as_array(res.keypoint_offsets, shape=(B + 1,)).copy()
        kp = np.zeros((0, 4), np.float32)
        dl = RECORD_FLOATS if self.record_output else DESC_LEN
        d = np.zeros((0, dl), np.float32) if self.params.estimate_descriptors else None
        if K > 0:
            kp = np.ctypeslib.as_array(C.cast(res.keypoints, C.POINTER(C.c_float)), shape=(K, 4))
            if res.descriptors:
                d = np.ctypeslib.as_array(C.cast(res.descriptors, C.POINTER(C.c_float)), shape=(K, dl))
            if copy:
                kp = kp.copy()
                d = d.copy() if d is not None else None
        return ko, kp, d


def imu_to_roll_pitch(quat_xyzw, cloud_leveling=True):
    """imuCallback (src:57-70): quaternion {x,y,z,w} -> (roll, pitch) as the node stores them."""
    q = np.ascontiguousarray(quat_xyzw, np.float64)
    r, p = C.c_double(0), C.c_double(0)
    st = N.lib().fe_imu_to_roll_pitch(_ptr(q), 1 if cloud_leveling else 0, C.byref(r), C.byref(p))
    if st != N.FE_OK:
        raise FeatureExtractionError(st, "fe_imu_to_roll_pitch")
    return float(r.value), float(p.value)


def rotation_matrix(roll, pitch):
    m = np.zeros(9, np.float32)
    N.lib().fe_rotation_matrix(float(roll), float(pitch), _ptr(m))
    return m.reshape(3, 3)


def pack_point_descriptors(keypoints, descriptors):
    """concatenateFields (src:119): (K, 1996) float32 pcl::PointDescriptor records."""
    kp = _cloud(keypoints)
    d = np.ascontiguousarray(descriptors, np.float32).reshape(len(kp), DESC_LEN)
    out = np.zeros((len(kp), N.RECORD_FLOATS), np.float32)
    st = N.lib().fe_pack_point_descriptors(_ptr(kp), _ptr(d), len(kp), _ptr(out))
    if st != N.FE_OK:
        raise FeatureExtractionError(st, "fe_pack_point_descriptors")
    return out


def debug_sort_replay(sizes):
    s = np.ascontiguousarray(sizes, np.int32)
    out = np.zeros(len(s), np.int32)
    N.lib().fe_debug_sort_replay(_ptr(s), len(s), _ptr(out))
    return out
