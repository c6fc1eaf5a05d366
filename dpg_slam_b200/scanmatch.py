"""Host-side mirror of the reference's scan-matching interface on top of the C ABI.

``ScanMatcher`` wraps one ``dpgicp_ctx`` (one GPU).  Method names follow the reference:

* :meth:`ScanMatcher.run_icp`            <-> ``DpgSLAM::runIcp``          (src/dpg_slam/dpg_slam.cc:362-446)
* :meth:`ScanMatcher.calculate_icp_cov`  <-> ``calculate_ICP_COV``        (src/icp_cov/cov_func_point_to_point.h:24)
* :meth:`ScanMatcher.submit_pairs`       <-> the loops that call runIcp   (dpg_slam.cc:79-107, 255-300)
* :meth:`ScanMatcher.enumerate_pairs`    <-> reoptimize's distance gate   (dpg_slam.cc:91-98)
* :func:`relative_guess`                 <-> ``math_utils::inverseTransformPoint`` (math_utils.cc:20-34)

Every compute call goes through ``libdpgicp.so``; a missing library or GPU raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np

from . import _abi
from ._abi import FACTOR_DTYPE, Params, Result, RESULT_DTYPE


class DpgIcpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"dpgicp error {code} ({_abi.ERRORS.get(code, '?')}): {msg}")
        self.code = code


def relative_guess(pose1, pose2) -> np.ndarray:
    """Pose of node_2 in node_1's frame as runIcp builds it (dpg_slam.cc:364-370,
    math_utils::inverseTransformPoint + AngleMod in float arithmetic).  pose = (x, y, theta)."""
    a = np.ascontiguousarray(pose1, np.float32)
    b = np.ascontiguousarray(pose2, np.float32)
    g = np.zeros(3, np.float32)
    rc = _abi.load_library().dpgicp_relative_guess(a.ctypes.data, b.ctypes.data, g.ctypes.data)
    if rc != 0:
        raise DpgIcpError(rc, "dpgicp_relative_guess")
    return g


def _pts(a) -> np.ndarray:
    a = np.ascontiguousarray(a, np.float32)
    if a.ndim != 2 or a.shape[1] not in (2, 4):
        raise ValueError("point clouds are (n, 2) packed xy or (n, 4) PointXYZ-layout float32 arrays")
    return a


class ScanMatcher:
    """One GPU's scan-matching context (device scan store + pair batch + kernels)."""

    def __init__(self, device: int = 0):
        self._lib = _abi.load_library()
        h = C.c_void_p()
        rc = self._lib.dpgicp_create(device, C.byref(h))
        if rc != 0:
            raise DpgIcpError(rc, (self._lib.dpgicp_last_error(None) or b"").decode())
        self._h = h
        self.device = device

    # ---- plumbing ---------------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise DpgIcpError(rc, (self._lib.dpgicp_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dpgicp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_stream(self, cuda_stream_handle: Optional[int]):
        """Run on an existing CUDA stream (e.g. ``torch.cuda.current_stream().cuda_stream``)."""
        self._check(self._lib.dpgicp_set_stream(self._h, C.c_void_p(cuda_stream_handle or 0)))

    def synchronize(self):
        self._check(self._lib.dpgicp_synchronize(self._h))

    # ---- scan store ---------------------------------------------------------------------------------
    def upload_scans(self, points: np.ndarray, offsets: np.ndarray):
        """CSR scan store: scan k = points[offsets[k]:offsets[k+1]] ((n,2) or (n,4) float32)."""
        pts = _pts(points) if len(points) else np.zeros((0, 2), np.float32)
        off = np.ascontiguousarray(offsets, np.int64)
        self._check(self._lib.dpgicp_upload_scans(self._h, pts.ctypes.data, pts.shape[1] * 4, off.ctypes.data,
                                                  off.shape[0] - 1))

    def upload_ranges(self, ranges: np.ndarray, scanner):
        """Raw range scans (n_scans, n_beams), converted on the device (createNode +
        getCachedPointCloudFromNode)."""
        r = np.ascontiguousarray(ranges, np.float32)
        self._check(self._lib.dpgicp_upload_ranges(self._h, r.ctypes.data, r.shape[0], r.shape[1],
                                                   scanner.angle_min, scanner.angle_max, scanner.range_max,
                                                   scanner.laser_x, scanner.laser_y, scanner.laser_theta))

    def append_scans(self, points: np.ndarray, offsets: np.ndarray):
        """Append CSR clouds (layout of :meth:`upload_scans`) as the next rows of the store; earlier rows, the pair
        batch and the node table stay.  A failed append leaves the store as it was."""
        pts = _pts(points) if len(points) else np.zeros((0, 2), np.float32)
        off = np.ascontiguousarray(offsets, np.int64)
        self._check(self._lib.dpgicp_append_scans(self._h, pts.ctypes.data, pts.shape[1] * 4, off.ctypes.data,
                                                  off.shape[0] - 1))

    def append_ranges(self, ranges: np.ndarray, scanner):
        """Append raw range scans (n_scans, n_beams) as the next rows of the store, converted on the device exactly as
        :meth:`upload_ranges` does (createNode: one call per new node).  A failed append leaves the store as it was."""
        r = np.ascontiguousarray(ranges, np.float32)
        self._check(self._lib.dpgicp_append_ranges(self._h, r.ctypes.data, r.shape[0], r.shape[1],
                                                   scanner.angle_min, scanner.angle_max, scanner.range_max,
                                                   scanner.laser_x, scanner.laser_y, scanner.laser_theta))

    def upload_ranges_ptr(self, host_ptr: int, n_scans: int, n_beams: int, scanner):
        """Same, from a raw (e.g. pinned) host pointer."""
        self._check(self._lib.dpgicp_upload_ranges(self._h, C.c_void_p(host_ptr), n_scans, n_beams,
                                                   scanner.angle_min, scanner.angle_max, scanner.range_max,
                                                   scanner.laser_x, scanner.laser_y, scanner.laser_theta))

    def upload_ranges_subset(self, ranges, scan_ids, scanner, n_scans_total: Optional[int] = None,
                             n_beams: Optional[int] = None):
        """Store row k = scan ``scan_ids[k]`` of ``ranges`` (an (n_scans, n_beams) float32 array, or a raw host
        pointer with ``n_scans_total``/``n_beams`` given).  Page-locked input is read in place by the kernel."""
        ids = np.ascontiguousarray(scan_ids, np.int32)
        if isinstance(ranges, int):
            ptr, total, beams = ranges, int(n_scans_total), int(n_beams)
        else:
            r = np.ascontiguousarray(ranges, np.float32)
            self._keep = r
            ptr, total, beams = r.ctypes.data, r.shape[0], r.shape[1]
        self._check(self._lib.dpgicp_upload_ranges_subset(self._h, C.c_void_p(ptr), total, beams, ids.ctypes.data, ids.shape[0],
                                                          scanner.angle_min, scanner.angle_max, scanner.range_max,
                                                          scanner.laser_x, scanner.laser_y, scanner.laser_theta))

    @property
    def scan_count(self) -> int:
        return int(self._lib.dpgicp_scan_count(self._h))

    def download_scan(self, k: int) -> np.ndarray:
        n = C.c_int32(_abi.MAX_POINTS)
        buf = np.zeros((_abi.MAX_POINTS, 2), np.float32)
        self._check(self._lib.dpgicp_download_scan(self._h, k, buf.ctypes.data, C.byref(n)))
        return np.ascontiguousarray(buf[:n.value])

    def download_store(self) -> Tuple[np.ndarray, np.ndarray]:
        clouds = [self.download_scan(k) for k in range(self.scan_count)]
        off = np.zeros(len(clouds) + 1, np.int64)
        off[1:] = np.cumsum([c.shape[0] for c in clouds])
        pts = np.concatenate(clouds) if clouds else np.zeros((0, 2), np.float32)
        return np.ascontiguousarray(pts, np.float32), off

    # ---- batched alignment -----------------------------------------------------------------------------
    def submit_pairs(self, src_idx, tgt_idx, guess, params: Params) -> np.ndarray:
        """Align every (source=node_2, target=node_1) pair; returns a RESULT_DTYPE record array."""
        s = np.ascontiguousarray(src_idx, np.int32)
        t = np.ascontiguousarray(tgt_idx, np.int32)
        g = np.ascontiguousarray(guess, np.float32).reshape(-1, 3)
        if not (s.shape[0] == t.shape[0] == g.shape[0]):
            raise ValueError("src_idx, tgt_idx and guess must have the same length")
        out = np.zeros(s.shape[0], RESULT_DTYPE)
        self._n_pairs = s.shape[0]
        self._check(self._lib.dpgicp_submit_pairs(self._h, s.ctypes.data, t.ctypes.data, g.ctypes.data, s.shape[0],
                                                  C.byref(params), out.ctypes.data))
        return out

    def set_pairs(self, src_idx, tgt_idx, guess):
        s = np.ascontiguousarray(src_idx, np.int32)
        t = np.ascontiguousarray(tgt_idx, np.int32)
        g = np.ascontiguousarray(guess, np.float32).reshape(-1, 3)
        self._n_pairs = s.shape[0]
        self._check(self._lib.dpgicp_set_pairs(self._h, s.ctypes.data, t.ctypes.data, g.ctypes.data, s.shape[0]))

    def set_pair_cost_hints(self, hints):
        """Expected relative cost per pair of the list set last (e.g. last time's ``iterations``): pairs are started
        in descending order so that long alignments do not start last.  ``None`` clears it."""
        if hints is None:
            self._check(self._lib.dpgicp_set_pair_cost_hints(self._h, None, 0))
            return
        h = np.ascontiguousarray(hints, np.float32)
        self._check(self._lib.dpgicp_set_pair_cost_hints(self._h, h.ctypes.data, h.shape[0]))

    def run(self, params: Params):
        """Launch the resident batch asynchronously on the context's stream."""
        self._check(self._lib.dpgicp_run(self._h, C.byref(params)))

    def run_range(self, params: Params, first: int, count: int):
        """Pairs [first, first + count) of the resident list (asynchronous)."""
        self._check(self._lib.dpgicp_run_range(self._h, C.byref(params), first, count))

    def fetch_results_range(self, first: int, count: int, host_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        if host_ptr is not None:
            self._check(self._lib.dpgicp_fetch_results_range(self._h, C.c_void_p(host_ptr), first, count))
            return None
        out = np.zeros(count, RESULT_DTYPE)
        self._check(self._lib.dpgicp_fetch_results_range(self._h, out.ctypes.data, first, count))
        return out

    def gather_fetch_range(self, first: int, count: int, host_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        if host_ptr is not None:
            self._check(self._lib.dpgicp_gather_fetch_range(self._h, C.c_void_p(host_ptr), first, count))
            return None
        out = np.zeros(count, RESULT_DTYPE)
        self._check(self._lib.dpgicp_gather_fetch_range(self._h, out.ctypes.data, first, count))
        return out

    def fetch_results(self, n: Optional[int] = None, out: Optional[np.ndarray] = None) -> np.ndarray:
        n = self._n_pairs if n is None else n
        if out is None:
            out = np.zeros(n, RESULT_DTYPE)
        self._check(self._lib.dpgicp_fetch_results(self._h, out.ctypes.data, n))
        return out

    def fetch_factors(self, n: Optional[int] = None) -> np.ndarray:
        """Records of the last run as pose-graph factors (``addObservationConstraint``, dpg_slam.cc:331-338):
        from/to node, Pose2 and the upper-triangular square-root information of the covariance."""
        n = self._n_pairs if n is None else n
        out = np.zeros(n, FACTOR_DTYPE)
        self._check(self._lib.dpgicp_fetch_factors(self._h, out.ctypes.data, n))
        return out

    def fetch_results_ptr(self, host_ptr: int, n: int):
        self._check(self._lib.dpgicp_fetch_results(self._h, C.c_void_p(host_ptr), n))

    def results_device_ptr(self) -> Tuple[int, int]:
        p, n = C.c_void_p(), C.c_int64()
        self._check(self._lib.dpgicp_results_device_ptr(self._h, C.byref(p), C.byref(n)))
        return int(p.value or 0), int(n.value)

    # ---- multi-GPU gather fused into the kernel epilogue (peer stores over NVLink) ------------------------------
    def gather_export(self, n_global_pairs: int) -> bytes:
        """Allocate this rank's buffer for the WHOLE batch's records; returns its 64-byte CUDA IPC handle."""
        h = (C.c_ubyte * _abi.IPC_HANDLE_BYTES)()
        self._check(self._lib.dpgicp_gather_export(self._h, n_global_pairs, C.byref(h)))
        return bytes(h)

    def gather_declare(self, n_global_pairs: int) -> bytes:
        """Root-only gathers: a rank other than 0 only declares the global batch size (placeholder buffer)."""
        h = (C.c_ubyte * _abi.IPC_HANDLE_BYTES)()
        self._check(self._lib.dpgicp_gather_declare(self._h, n_global_pairs, C.byref(h)))
        return bytes(h)

    def gather_attach(self, handles, rank: int):
        """``handles``: every rank's exported handle, in rank order.  From now on ``run`` stores record k of the
        local shard into slot ``rank + k * world`` of every rank's buffer."""
        blob = b"".join(handles)
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self._check(self._lib.dpgicp_gather_attach(self._h, C.byref(buf), len(handles), rank))

    def gather_detach(self):
        self._check(self._lib.dpgicp_gather_detach(self._h))

    def gather_fetch(self, n_global_pairs: int) -> np.ndarray:
        out = np.zeros(n_global_pairs, RESULT_DTYPE)
        self._check(self._lib.dpgicp_gather_fetch(self._h, out.ctypes.data, n_global_pairs))
        return out

    def last_run_counters(self) -> dict:
        c = (C.c_uint64 * 8)()
        self._check(self._lib.dpgicp_last_run_counters(self._h, C.byref(c)))
        return {"iterations": int(c[0]), "correspondences": int(c[1]), "distance_evals": int(c[2]),
                "box_tests": int(c[3]), "kernel_launches": int(c[4]),
                "dev_candidates": int(c[5]), "dev_loose_searches": int(c[6]), "dev_searches": int(c[7])}

    def fp32_probe(self) -> dict:
        """Measured FP32 CUDA-core rates of this GPU (ops/s): separately rounded FMUL+FADD and FFMA."""
        a, b = C.c_double(0), C.c_double(0)
        self._check(self._lib.dpgicp_fp32_probe(self._h, C.byref(a), C.byref(b)))
        p = C.c_double(0)
        self._check(self._lib.dpgicp_fp32x2_probe(self._h, C.byref(p)))
        return {"mul_add_ops_per_s": a.value, "fma_ops_per_s": b.value, "mul_add_packed_ops_per_s": p.value}

    # ---- the two reference call shapes ----------------------------------------------------------------
    def run_icp(self, node_1_cloud, node_2_cloud, guess, params: Optional[Params] = None):
        """``runIcp(node_1, node_2, icp_results)``: aligns node_2's cloud (source) onto node_1's
        (target) from ``guess`` = pose of node_2 in node_1's frame (use :func:`relative_guess`).
        Returns ``(converged, ((tx, ty), theta), cov3x3, record)`` — converged is what
        ``icp.hasConverged()`` returns (dpg_slam.cc:445)."""
        p = params or Params.defaults()
        s, t = _pts(node_2_cloud), _pts(node_1_cloud)
        if s.shape[1] != t.shape[1]:
            raise ValueError("both clouds must use the same point layout")
        g = np.ascontiguousarray(guess, np.float32)
        res = Result()
        self._check(self._lib.dpgicp_single_pair(self._h, s.ctypes.data, s.shape[0], t.ctypes.data, t.shape[0],
                                                 s.shape[1] * 4, g.ctypes.data, C.byref(p), C.byref(res)))
        converged = bool(res.status & _abi.FLAG_CONVERGED)
        cov = np.array(res.cov, np.float64).reshape(3, 3)
        return converged, ((res.tx, res.ty), res.theta), cov, res

    def calculate_icp_cov(self, data_pi, model_qi, transform4x4, params: Optional[Params] = None):
        """``calculate_ICP_COV(data_pi, model_qi, transform, ICP_COV, sx2, sy2, st2)``; the three
        variances travel in ``params``.  Returns ``(cov3x3, status)``."""
        p = params or Params.defaults()
        a, b = _pts(data_pi), _pts(model_qi)
        T = np.asarray(transform4x4, np.float32).reshape(4, 4)
        Tc = np.ascontiguousarray(T.T).reshape(16)          # column-major, as Eigen::Matrix4f stores it
        cov = np.zeros(9, np.float64)
        st = C.c_uint32(0)
        self._check(self._lib.dpgicp_cov(self._h, a.ctypes.data, a.shape[0], b.ctypes.data, b.shape[0], a.shape[1] * 4,
                                         Tc.ctypes.data, C.byref(p), cov.ctypes.data, C.byref(st)))
        return cov.reshape(3, 3), int(st.value)

    def calculate_icp_cov_pairs(self, data_idx, model_idx, T, params: Optional[Params] = None):
        """Batched ``calculate_ICP_COV`` over the scan store: item k pairs scans ``data_idx[k]`` / ``model_idx[k]`` by
        index under ``T[k] = (T00, T10, T03, T13)``.  Returns ``(cov (n, 3, 3), status (n,), kernel_ms)``."""
        p = params or Params.defaults()
        a = np.ascontiguousarray(data_idx, np.int32)
        b = np.ascontiguousarray(model_idx, np.int32)
        t = np.ascontiguousarray(T, np.float32).reshape(-1, 4)
        cov = np.zeros((a.shape[0], 9), np.float64)
        st = np.zeros(a.shape[0], np.uint32)
        ms = C.c_float(0)
        self._check(self._lib.dpgicp_cov_pairs(self._h, a.ctypes.data, b.ctypes.data, t.ctypes.data, a.shape[0], C.byref(p),
                                               cov.ctypes.data, st.ctypes.data, C.byref(ms)))
        return cov.reshape(-1, 3, 3), st, float(ms.value)

    # ---- parity hook + callers' gate ---------------------------------------------------------------------
    def correspondences(self, source_ds, target_ds, T, params: Params):
        """One correspondence pass at iterate T = (c, s, tx, ty) -> (corr_tgt int32, d2 float32)."""
        s, t = _pts(source_ds), _pts(target_ds)
        Tm = np.ascontiguousarray(T, np.float32)
        corr = np.full(max(s.shape[0], 1), -1, np.int32)
        d2 = np.zeros(max(s.shape[0], 1), np.float32)
        self._check(self._lib.dpgicp_correspondences(self._h, s.ctypes.data, s.shape[0], t.ctypes.data, t.shape[0],
                                                     s.shape[1] * 4, Tm.ctypes.data, C.byref(params),
                                                     corr.ctypes.data, d2.ctypes.data))
        return corr[:s.shape[0]], d2[:s.shape[0]]

    def correspondences_seeded(self, source_ds, target_ds, T, params: Params, prev_nn):
        """The same pass with the sticky tie preference of an ICP run in progress: ``prev_nn[i]`` = forward neighbour
        of source point i in the previous pass (-1 = none).  Returns (corr_tgt, d2, nn_out)."""
        s, t = _pts(source_ds), _pts(target_ds)
        Tm = np.ascontiguousarray(T, np.float32)
        n = max(s.shape[0], 1)
        corr = np.full(n, -1, np.int32)
        d2 = np.zeros(n, np.float32)
        nn = np.full(n, -1, np.int32)
        prev = np.ascontiguousarray(prev_nn, np.int32)
        self._check(self._lib.dpgicp_correspondences_seeded(self._h, s.ctypes.data, s.shape[0], t.ctypes.data, t.shape[0],
                                                            s.shape[1] * 4, Tm.ctypes.data, C.byref(params),
                                                            prev.ctypes.data, corr.ctypes.data, d2.ctypes.data, nn.ctypes.data))
        return corr[:s.shape[0]], d2[:s.shape[0]], nn[:s.shape[0]]

    # ---- device-resident callers: nodes in, pair batch left on the device ------------------------------------
    def set_nodes(self, node_poses, node_pass):
        """Pose-graph node estimates (n, 3) = (x, y, theta) and pass numbers; node k owns scan k of the store."""
        ps = np.ascontiguousarray(node_poses, np.float32).reshape(-1, 3)
        pa = np.ascontiguousarray(node_pass, np.int32)
        if ps.shape[0] != pa.shape[0]:
            raise ValueError("node_poses and node_pass must have the same length")
        self._check(self._lib.dpgicp_set_nodes(self._h, ps.ctypes.data, pa.ctypes.data, ps.shape[0]))

    def enumerate_pairs_device(self, mode=_abi.ENUM_REOPTIMIZE, same_pass_radius=5.0, other_pass_radius=2.0,
                               shard_rank=0, shard_world=1) -> Tuple[int, int]:
        """Build the caller's pair list (``reoptimize`` or ``updatePoseGraphObsConstraints``) and every pair's guess on
        the device, in the reference's loop order; this context keeps the pairs with global index % world == rank as
        its batch.  Returns (n_pairs_total, n_pairs_local)."""
        tot, loc = C.c_int64(0), C.c_int64(0)
        self._check(self._lib.dpgicp_enumerate_pairs_device(self._h, mode, same_pass_radius, other_pass_radius,
                                                            shard_rank, shard_world, C.byref(tot), C.byref(loc)))
        self._n_pairs = int(loc.value)
        return int(tot.value), int(loc.value)

    def fetch_pairs(self, n: Optional[int] = None):
        """The current batch's pair list: (src_idx, tgt_idx, T (n, 4) = guess entries c, s, tx, ty)."""
        n = self._n_pairs if n is None else n
        src = np.zeros(n, np.int32)
        tgt = np.zeros(n, np.int32)
        T = np.zeros((n, 4), np.float32)
        self._check(self._lib.dpgicp_fetch_pairs(self._h, src.ctypes.data, tgt.ctypes.data, T.ctypes.data, n))
        return src, tgt, T

    def convert_ranges_device(self, device_ptr: int, n_scans: int, n_beams: int, scanner):
        """Scan store from raw ranges already in device memory (e.g. all-gathered there over NCCL)."""
        self._check(self._lib.dpgicp_convert_ranges_device(self._h, C.c_void_p(device_ptr), n_scans, n_beams,
                                                           scanner.angle_min, scanner.angle_max, scanner.range_max,
                                                           scanner.laser_x, scanner.laser_y, scanner.laser_theta))

    def gather_set_root_only(self, root_only: bool):
        self._check(self._lib.dpgicp_gather_set_root_only(self._h, int(bool(root_only))))

    def enable_stage_timing(self, on: bool = True):
        self._check(self._lib.dpgicp_enable_stage_timing(self._h, int(bool(on))))

    def last_run_stage_ms(self):
        ms = (C.c_float * 8)()
        n = C.c_int32(0)
        self._check(self._lib.dpgicp_last_run_stage_ms(self._h, C.byref(ms), C.byref(n)))
        return [float(ms[k]) for k in range(n.value)]

    def enumerate_pairs(self, node_xy, node_pass, same_pass_radius=5.0, other_pass_radius=2.0):
        """Pair list of one ``reoptimize()`` in the reference's loop order (parameters.h:212,224)."""
        xy = np.ascontiguousarray(node_xy, np.float32)
        ps = np.ascontiguousarray(node_pass, np.int32)
        n = C.c_int64(0)
        rc = self._lib.dpgicp_enumerate_pairs(self._h, xy.ctypes.data, ps.ctypes.data, xy.shape[0], same_pass_radius,
                                              other_pass_radius, None, None, C.byref(n))
        if rc not in (0, -7):
            self._check(rc)
        src = np.zeros(n.value, np.int32)
        tgt = np.zeros(n.value, np.int32)
        if n.value:
            self._check(self._lib.dpgicp_enumerate_pairs(self._h, xy.ctypes.data, ps.ctypes.data, xy.shape[0],
                                                         same_pass_radius, other_pass_radius, src.ctypes.data,
                                                         tgt.ctypes.data, C.byref(n)))
        return src, tgt
