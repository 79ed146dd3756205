"""Seeded synthetic VLP-16 scans (SURVEY.md §8d) — ctypes binding of synth/libfe_synth.so.

Input generator for the parity tests and bench.py; host only, not part of the hot path.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "synth")
_LIB = None


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def _lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "libfe_synth.so")
        if not os.path.exists(path):
            build()
        _LIB = C.CDLL(path)
    return _LIB


def default_azimuth_steps(config):
    return int(_lib().fes_default_azimuth_steps(C.c_int(config)))


def generate(config, n_scans, scan_index_base=0, azimuth_steps=0, n_threads=0, out=None):
    """-> points (N,4) float32, scan_offsets (n_scans+1,) int64, roll_pitch (n_scans,2) float64.

    config: 1..5 as in BASELINE.json `configs` (5 uses config 2's generator).
    `out`: optional preallocated (cap,4) float32 array (e.g. pinned memory) to generate into.
    """
    A = azimuth_steps or default_azimuth_steps(config)
    cap = 16 * A * n_scans
    if out is None:
        out = np.empty((max(cap, 1), 4), np.float32)
    else:
        assert out.dtype == np.float32 and out.flags.c_contiguous
        cap = min(cap, out.shape[0])
    offs = np.zeros(n_scans + 1, np.int64)
    rp = np.zeros((max(n_scans, 1), 2), np.float64)
    if n_threads <= 0:
        n_threads = len(os.sched_getaffinity(0))
    st = _lib().fes_generate(C.c_int(config), C.c_int64(scan_index_base), C.c_int(n_scans), C.c_int(A),
                             C.c_int(n_threads), out.ctypes.data_as(C.c_void_p), C.c_int64(cap),
                             offs.ctypes.data_as(C.c_void_p), rp.ctypes.data_as(C.c_void_p))
    if st != 0:
        raise RuntimeError("fes_generate: capacity too small")
    return out[: offs[-1]], offs, rp[:n_scans]


def generate_poses(config, scene_index, poses, azimuth_steps=0, n_threads=0):
    """One scene seen from several sensor poses: the scene of generate()'s scan `scene_index`, rendered from each
    poses[s] = (x, y, yaw) of the scene frame (metres, radians).  Scan 0 at pose (0, 0, 0) is generate()'s scan
    `scene_index` byte for byte; scans s >= 1 draw roll, pitch and noise from a stream of their own.
    -> points (N,4) float32, scan_offsets (n_scans+1,) int64, roll_pitch (n_scans,2) float64."""
    poses = np.ascontiguousarray(poses, np.float64).reshape(-1, 3)
    n_scans = len(poses)
    A = azimuth_steps or default_azimuth_steps(config)
    cap = 16 * A * n_scans
    out = np.empty((max(cap, 1), 4), np.float32)
    offs = np.zeros(n_scans + 1, np.int64)
    rp = np.zeros((max(n_scans, 1), 2), np.float64)
    if n_threads <= 0:
        n_threads = len(os.sched_getaffinity(0))
    st = _lib().fes_generate_poses(C.c_int(config), C.c_int64(scene_index), C.c_int(n_scans), C.c_int(A),
                                   C.c_int(n_threads), poses.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                   C.c_int64(cap), offs.ctypes.data_as(C.c_void_p), rp.ctypes.data_as(C.c_void_p))
    if st != 0:
        raise RuntimeError("fes_generate_poses: capacity too small")
    return out[: offs[-1]], offs, rp[:n_scans]
