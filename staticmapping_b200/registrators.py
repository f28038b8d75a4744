"""Host-side mirror of the reference's plugin surface, registrator::Interface
(/root/reference/registrators/interface.h:67-119), over the C ABI of libsm_b200.so.

Same member names, argument meaning and error behaviour as the reference:

* ``CreateMatcher(options)``            interface.cc:139-173
* ``Interface.InitWithXml(node)``       interface.cc:62-90  (unknown <param> -> CheckFailure,
                                         the reference glog-CHECK-aborts)
* ``SetInputSource / SetInputTarget``   icp_fast.cc:421-431 (deep copy; target needs normals)
* ``Align(guess) -> (ok, result)``      icp_fast.cc:455-529 (C++: bool Align(guess, result&))
* ``GetFitnessScore / GetType / PrintOptions / Enable/DisableInnerCompensation``

Clouds are passed as the data the reference's ``InnerPointCloudData`` holds for each
matcher: an ``EigenCloud`` (double points [+ normals]) for IcpFast.
"""
from __future__ import annotations

import ctypes as C
import enum
import xml.etree.ElementTree as ET
from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import _lib


class Type(enum.IntEnum):
    """registrator::Type (interface.h:41-50)."""
    kNoType = 0
    kIcpPM = 1
    kLibicp = 2
    kNdtWithGicp = 3
    kLegoLoam = 4
    kNdt = 5
    kFastIcp = 6


class CheckFailure(RuntimeError):
    """Raised where the reference would glog CHECK-fail (abort)."""


@dataclass
class EigenCloud:
    """data::EigenPointCloud (cloud_types.h:121-147): (N,3) float64 points, optional normals.
    C-contiguous (N,3) == Eigen's 3xN column-major storage."""
    points: np.ndarray
    normals: Optional[np.ndarray] = None

    def __post_init__(self):
        self.points = np.ascontiguousarray(np.asarray(self.points, dtype=np.float64))
        if self.points.ndim != 2 or self.points.shape[1] != 3:
            raise ValueError("points must be (N,3)")
        if self.normals is not None:
            self.normals = np.ascontiguousarray(np.asarray(self.normals, dtype=np.float64))
            if self.normals.shape != self.points.shape:
                raise ValueError("normals must match points")

    def HasNormals(self):
        return self.normals is not None and self.normals.shape[0] > 0

    @staticmethod
    def FromPointCloud(xyz_f32):
        """EigenPointCloud::FromPointCloud (cloud_types.cc:328-345): float AoS -> double."""
        return EigenCloud(np.asarray(xyz_f32, dtype=np.float32).astype(np.float64))


@dataclass
class InnerCloud:
    """data::InnerCloudType (cloud_types.h:59-77): the float cloud `Ndt` / `NdtWithGicp` keep
    (x, y, z of InnerPointType; intensity / factor are not used by the matchers).
    points: (N,3) float32, or (N,5) float32 rows laid out like InnerPointType (20-byte stride)."""
    points: np.ndarray

    def __post_init__(self):
        self.points = np.ascontiguousarray(np.asarray(self.points, dtype=np.float32))
        if self.points.ndim != 2 or self.points.shape[1] not in (3, 5):
            raise ValueError("points must be (N,3) or (N,5) float32")

    def Empty(self):
        return self.points.shape[0] == 0

    @property
    def stride_bytes(self):
        return 4 * self.points.shape[1]


@dataclass
class MatcherOptions:
    """registrator::MatcherOptions (interface.h:59-65)."""
    type: Type = Type.kIcpPM
    accepted_min_score: float = 0.7
    registrator_options_node: Optional[object] = None   # xml string / Element / dict
    inner_filters_node: Optional[object] = None


def _params_from_node(node):
    if node is None:
        return []
    if isinstance(node, dict):
        return [(k, str(v)) for k, v in node.items()]
    if isinstance(node, (str, bytes)):
        node = ET.fromstring(node)
    return [(p.attrib.get("name", ""), (p.text or "").strip()) for p in node.findall("param")]


class Interface:
    """registrator::Interface.  One instance is used by one thread at a time; distinct
    instances may run concurrently (each owns a CUDA stream + workspace)."""

    _type = Type.kNoType

    def __init__(self, device: int = 0):
        self._lib = _lib.lib()
        self._h = C.c_void_p()
        rc = self._lib.sm_create(int(self._type), device, C.byref(self._h))
        if rc == -20:
            raise RuntimeError("staticmapping_b200: no CUDA device visible and there is no CPU "
                               "fallback (SM_ERR_NO_DEVICE)")
        if rc != 0:
            raise RuntimeError(f"sm_create failed with {rc}")
        self._inner_compensation = False
        self._source = None
        self._target = None

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.sm_destroy(h)
            self._h = C.c_void_p()

    def _check(self, rc, what):
        if rc < 0:
            msg = self._lib.sm_last_error(self._h)
            raise CheckFailure(f"{what}: {msg.decode() if msg else rc} (code {rc})")
        return rc

    # --- options -------------------------------------------------------------------------
    def InitWithXml(self, node):
        for name, text in _params_from_node(node):
            self._check(self._lib.sm_set_option(self._h, name.encode(), text.encode()),
                        "InitWithXml")

    def InitInnerFiltersWithXml(self, node):
        return None  # interface.cc:92-113: a TODO in the reference, no effect

    def InitWithOptions(self):
        return None

    def PrintOptions(self):
        buf = C.create_string_buffer(4096)
        self._lib.sm_print_options(self._h, buf, 4096)
        text = buf.value.decode()
        print(text, end="")
        return text

    def EnableInnerCompensation(self):
        self._inner_compensation = True   # no caller in the reference (SURVEY Appendix A)

    def DisableInnerCompensation(self):
        self._inner_compensation = False

    # --- data ----------------------------------------------------------------------------
    def SetInputSource(self, cloud: EigenCloud):
        raise NotImplementedError

    def SetInputTarget(self, cloud: EigenCloud):
        raise NotImplementedError

    def Align(self, guess):
        """Returns (ok, result 4x4).  C++: bool Align(const Matrix4d& guess, Matrix4d& result)."""
        g = np.ascontiguousarray(np.asarray(guess, dtype=np.float64).T).ravel()
        res = np.zeros(16, dtype=np.float64)
        rc = self._check(self._lib.sm_align(self._h, g.ctypes.data_as(_lib._DP),
                                            res.ctypes.data_as(_lib._DP)), "Align")
        return bool(rc), res.reshape(4, 4).T.copy()

    def AlignAsync(self, guess):
        """First half of Align: enqueue and return (engine extension, see sm_align_async)."""
        g = np.ascontiguousarray(np.asarray(guess, dtype=np.float64).T).ravel()
        self._check(self._lib.sm_align_async(self._h, g.ctypes.data_as(_lib._DP)), "AlignAsync")

    def AlignWait(self):
        """Second half of Align: returns (ok, result 4x4)."""
        res = np.zeros(16, dtype=np.float64)
        rc = self._check(self._lib.sm_align_wait(self._h, res.ctypes.data_as(_lib._DP)), "AlignWait")
        return bool(rc), res.reshape(4, 4).T.copy()

    def GetFitnessScore(self):
        return float(self._lib.sm_get_fitness_score(self._h))

    def GetType(self):
        return Type(self._lib.sm_get_type(self._h))

    def SetStream(self, cuda_stream: int = 0):
        """Run on the caller's CUDA stream (0 / None -> the handle's own stream)."""
        self._check(self._lib.sm_set_stream(self._h, cuda_stream or None), "SetStream")

    def GetAlignInfo(self):
        info = _lib.AlignInfo()
        self._lib.sm_get_align_info(self._h, C.byref(info))
        out = {k: getattr(info, k) for k, _ in _lib.AlignInfo._fields_ if k not in ("reserved", "aux")}
        out["aux"] = [float(v) for v in info.aux]
        return out


class IcpFast(Interface):
    """registrator::IcpFast (icp_fast.h:37-62)."""
    _type = Type.kFastIcp

    def SetInputSource(self, cloud: EigenCloud):
        if cloud is None or cloud.points.shape[0] == 0:
            raise CheckFailure("SetInputSource: CHECK(cloud) failed (icp_fast.cc:422-423)")
        self._check(self._lib.sm_set_input_source(self._h, cloud.points.ctypes.data,
                                                  cloud.points.shape[0]), "SetInputSource")

    def SetInputTarget(self, cloud: EigenCloud):
        if cloud is None or cloud.points.shape[0] == 0:
            raise CheckFailure("SetInputTarget: CHECK(cloud) failed (icp_fast.cc:428-429)")
        if not cloud.HasNormals():
            raise CheckFailure("SetInputTarget: CHECK(HasNormals()) failed (icp_fast.cc:430)")
        self._check(self._lib.sm_set_input_target(self._h, cloud.points.ctypes.data,
                                                  cloud.normals.ctypes.data,
                                                  cloud.points.shape[0]), "SetInputTarget")

    # device-resident variants (pointers to 3xN column-major doubles in this GPU's memory)
    def SetInputSourceDevice(self, dev_ptr: int, n: int):
        self._check(self._lib.sm_set_input_source_device(self._h, dev_ptr, n), "SetInputSource")

    def SetInputTargetDevice(self, dev_points: int, dev_normals: int, n: int):
        self._check(self._lib.sm_set_input_target_device(self._h, dev_points, dev_normals, n),
                    "SetInputTarget")


class Ndt(Interface):
    """registrator::Ndt (ndt.h / ndt.cc:28-64): pclomp NDT, resolution 1.0, KDTREE neighbour
    search.  GetFitnessScore() is PCL's mean squared NN distance (LOWER is better), unlike the
    ICP matchers' exp(-distance) (SURVEY 3.4)."""
    _type = Type.kNdt

    def InitWithXml(self, node):
        # Ndt registers no option (ndt.cc:28-34): any <param> hits the CHECK in interface.cc:66
        for name, _ in _params_from_node(node):
            raise CheckFailure(f"Init an unknown option of this matcher! ({name})")

    def SetEngineOptions(self, **kw):
        """pclomp setters the reference hard-codes (resolution, step_size, outlier_ratio,
        transformation_epsilon, max_iterations); not reachable from the reference's XML."""
        for k, v in kw.items():
            self._check(self._lib.sm_set_option(self._h, k.encode(), str(v).encode()), "option")

    def SetInputSource(self, cloud: InnerCloud):
        # Interface::SetInputSource (interface.cc:38-48): null resets, empty only warns
        self._source = None
        if cloud is None:
            return
        if cloud.Empty():
            print("cloud is empty.")
            return
        self._check(self._lib.sm_set_input_source_f32(self._h, cloud.points.ctypes.data,
                                                      cloud.points.shape[0], cloud.stride_bytes),
                    "SetInputSource")
        self._source = cloud

    def SetInputTarget(self, cloud: InnerCloud):
        self._target = None
        if cloud is None:
            return
        if cloud.Empty():
            print("cloud is empty.")
            return
        self._check(self._lib.sm_set_input_target_f32(self._h, cloud.points.ctypes.data,
                                                      cloud.points.shape[0], cloud.stride_bytes),
                    "SetInputTarget")
        self._target = cloud

    def Align(self, guess):
        if self._source is None or self._target is None:   # ndt.cc:40-42
            return False, np.asarray(guess, dtype=np.float64).copy()
        return super().Align(guess)


class NdtWithGicp(Ndt):
    """registrator::NdtWithGicp (ndt_gicp.h / ndt_gicp.cc:28-112): ApproximateVoxelGrid(0.2 m) on
    both clouds -> stock PCL NDT (resolution 1.0, step 0.1, eps 0.01, 35 it) -> stock PCL GICP
    (rotation eps 1e-3, 35 it), gated on NDT fitness <= 1.  GetFitnessScore() = exp(-GICP fitness).
    Registered options (ndt_gicp.cc:31-36): use_ndt, using_voxel_filter, voxel_resolution."""
    _type = Type.kNdtWithGicp

    def InitWithXml(self, node):
        Interface.InitWithXml(self, node)

    def Align(self, guess):
        if self._source is None or self._target is None:
            raise CheckFailure("NdtWithGicp::Align: input cloud not set (null dereference in the reference)")
        return Interface.Align(self, guess)


class IcpUsingPointMatcher(Ndt):
    """Stand-in for registrator::IcpUsingPointMatcher (icp_pointmatcher.h / .cc:125-247), the
    libpointmatcher-driven ICP that loop_detector.cc:304-308 constructs directly.  Same module
    chain as the reference's default config (:166-247): reading filter RandomSampling 0.9,
    reference filter SamplingSurfaceNormal knn 7 (== CalculateNormals), k-d tree matcher eps 3.16,
    TrimmedDist 0.7, point-to-plane minimiser, 150-iteration counter + 4-sample differential
    checker; GetFitnessScore() = exp(-mean kept distance) of the UNFILTERED clouds re-matched after
    the result (:131-148), Align() is False below 0.6 (:145).
    libpointmatcher itself (1.3.1, float, std::rand) is external to the reference tree, so this is
    a deterministic double-precision equivalent built from the IcpFast kernels, not a bit-level
    restatement.  It registers no XML option (the reference takes a YAML file name instead)."""
    _type = Type.kIcpPM

    def __init__(self, device: int = 0, ymal_file: str = ""):
        if ymal_file:
            raise CheckFailure("IcpUsingPointMatcher: YAML configs are not supported, only loadDefaultConfig()")
        super().__init__(device)

    def Align(self, guess):
        if self._source is None or self._target is None:
            raise CheckFailure("IcpUsingPointMatcher::Align: input cloud not set")
        return Interface.Align(self, guess)


def CreateMatcher(options: MatcherOptions, verbose: bool = False, device: int = 0) -> Interface:
    """registrator::CreateMatcher (interface.cc:139-173)."""
    t = Type(options.type)
    if t == Type.kFastIcp:
        matcher = IcpFast(device)
    elif t in (Type.kLibicp, Type.kLegoLoam):
        raise CheckFailure("The registrator using libicp & lego-loam is deprecated. "
                           "please choose another type")   # LOG(FATAL), interface.cc:154-157
    elif t == Type.kNdt:
        matcher = Ndt(device)
    elif t == Type.kNdtWithGicp:
        matcher = NdtWithGicp(device)
    elif t == Type.kIcpPM:
        matcher = IcpUsingPointMatcher(device)
    else:
        print("Wrong type")   # PRINT_ERROR + nullptr, interface.cc:158-160
        return None
    if options.registrator_options_node is not None:
        matcher.InitWithXml(options.registrator_options_node)
    if verbose:
        matcher.PrintOptions()
    matcher.InitWithOptions()
    return matcher


def AlignBatch(matchers, guesses):
    """Batched Align over matcher instances whose inputs are set (sm_align_batch): what
    loop_detector.cc:216-228 / map_builder.cc:706-708 do with a thread pool, from one host thread.
    Returns (oks, results) with results of shape (n, 4, 4)."""
    n = len(matchers)
    lib = _lib.lib()
    hs = (C.c_void_p * n)(*[m._h for m in matchers])
    g = np.ascontiguousarray(np.stack([np.asarray(x, dtype=np.float64).T for x in guesses]).reshape(n, 16))
    res = np.zeros((n, 16), dtype=np.float64)
    rcs = np.zeros(n, dtype=np.int32)
    lib.sm_align_batch(hs, n, g.ctypes.data, res.ctypes.data, rcs.ctypes.data)
    for m, rc in zip(matchers, rcs):
        m._check(int(rc), "AlignBatch")
    return [bool(r) for r in rcs], res.reshape(n, 4, 4).transpose(0, 2, 1).copy()


def AlignPairs(matchers, pairs):
    """n_pairs independent IcpFast alignments pipelined over the given instances (sm_align_pairs).
    `pairs`: sequence of dicts {source, target, normals, guess (optional), on_device (optional)} where
    the clouds are (N, 3) float64 C-contiguous arrays (host; pinned memory overlaps best) or, with
    on_device, integer device pointers plus n_source / n_target.
    Returns (rcs, results (n, 4, 4), scores (n,))."""
    n = len(pairs)
    lib = _lib.lib()
    hs = (C.c_void_p * len(matchers))(*[m._h for m in matchers])
    arr = (_lib.Pair * n)()
    keep = []
    for k, pr in enumerate(pairs):
        dev = bool(pr.get("on_device", False))
        if dev:
            arr[k].source, arr[k].target, arr[k].target_normals = pr["source"], pr["target"], pr["normals"]
            arr[k].n_source, arr[k].n_target = int(pr["n_source"]), int(pr["n_target"])
        else:
            src, tgt, nrm = pr["source"], pr["target"], pr["normals"]
            arr[k].source, arr[k].target, arr[k].target_normals = _ptr(src), _ptr(tgt), _ptr(nrm)
            arr[k].n_source = int(pr["n_source"]) if "n_source" in pr else len(src)
            arr[k].n_target = int(pr["n_target"]) if "n_target" in pr else len(tgt)
        g = pr.get("guess")
        if g is not None:
            g = np.ascontiguousarray(np.asarray(g, dtype=np.float64).T).ravel()
            keep.append(g)
            arr[k].guess = g.ctypes.data
        arr[k].on_device = 1 if dev else 0
    res = np.zeros((n, 16), dtype=np.float64)
    scores = np.zeros(n, dtype=np.float64)
    rcs = np.zeros(n, dtype=np.int32)
    rc = lib.sm_align_pairs(hs, len(matchers), arr, n, res.ctypes.data, scores.ctypes.data, rcs.ctypes.data)
    if rc == -11:
        raise CheckFailure("AlignPairs: IcpFast instances only")
    for k, r in enumerate(rcs):
        matchers[k % len(matchers)]._check(int(r), "AlignPairs")
    return rcs, res.reshape(n, 4, 4).transpose(0, 2, 1).copy(), scores


def _ptr(a):
    """address of a float64 (N, 3) C-contiguous numpy array or torch tensor (data_ptr), or an int"""
    if isinstance(a, int):
        return a
    if hasattr(a, "data_ptr"):
        return int(a.data_ptr())
    a = np.asarray(a)
    if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"]:
        raise ValueError("AlignPairs needs C-contiguous float64 clouds (no hidden copies: the engine reads them asynchronously)")
    return a.ctypes.data


def knn1(target, query, epsilon=3.16, bucket_size=8, device=0, queries_per_cta=0):
    """libnabo-compatible 1-NN on the GPU (NNS::create + knn, icp_fast.cc:466-467,177-178).
    queries_per_cta > 0: the test hook sm_debug_knn1_batched (the launch shape of batched alignments)."""
    lib = _lib.lib()
    t = np.ascontiguousarray(np.asarray(target, dtype=np.float64))
    q = np.ascontiguousarray(np.asarray(query, dtype=np.float64))
    ids = np.empty(q.shape[0], dtype=np.int32)
    d2 = np.empty(q.shape[0], dtype=np.float64)
    if queries_per_cta:
        rc = lib.sm_debug_knn1_batched(device, t.ctypes.data, t.shape[0], q.ctypes.data, q.shape[0], float(epsilon),
                                       int(bucket_size), int(queries_per_cta), ids.ctypes.data, d2.ctypes.data)
    else:
        rc = lib.sm_knn1(device, t.ctypes.data, t.shape[0], q.ctypes.data, q.shape[0], float(epsilon),
                         int(bucket_size), ids.ctypes.data, d2.ctypes.data)
    if rc == -20:
        raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
    if rc != 0:
        raise RuntimeError(f"sm_knn1 failed with {rc}")
    return ids, d2


def CalculateNormals(points, device=0) -> EigenCloud:
    """EigenPointCloud::CalculateNormals on the GPU (cloud_types.cc:347-368): returns the
    decimated cloud (one mean point + unit normal per valid <=7-point leaf)."""
    lib = _lib.lib()
    p = np.ascontiguousarray(np.asarray(points, dtype=np.float64))
    out_p = np.empty_like(p)
    out_n = np.empty_like(p)
    m = C.c_int64(0)
    rc = lib.sm_calculate_normals(device, p.ctypes.data, p.shape[0], out_p.ctypes.data,
                                  out_n.ctypes.data, C.byref(m))
    if rc == -20:
        raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
    if rc != 0:
        raise RuntimeError(f"sm_calculate_normals failed with {rc}")
    return EigenCloud(out_p[:m.value].copy(), out_n[:m.value].copy())


def MotionCompensation(raw_cloud, delta_transform, device=0):
    """MotionCompensation (builder/map_builder.cc:232-257) on the GPU.  `raw_cloud` is an (N,5)
    float32 array of InnerPointType rows (x, y, z, intensity, factor); every point is moved by
    common::InterpolateTransform(Identity, delta, factor) (common/math.h:198-211).  Raises
    CheckFailure where the reference CHECK-fails (a factor outside [0, 1])."""
    lib = _lib.lib()
    pts = np.ascontiguousarray(np.asarray(raw_cloud, dtype=np.float32))
    if pts.ndim != 2 or pts.shape[1] != 5:
        raise ValueError("raw_cloud must be (N,5): x, y, z, intensity, factor")
    d = np.asfortranarray(np.asarray(delta_transform, dtype=np.float64))
    if d.shape != (4, 4):
        raise ValueError("delta_transform must be 4x4")
    out = np.empty_like(pts)
    rc = lib.sm_motion_compensation(device, pts.ctypes.data, pts.shape[0], 20, d.ctypes.data_as(_lib._DP),
                                    out.ctypes.data)
    if rc == -20:
        raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
    if rc == -1:
        raise CheckFailure("Check failed: factor >= 0. && factor <= 1. (common/math.h:201)")
    if rc != 0:
        raise RuntimeError(f"sm_motion_compensation failed with {rc}")
    return out


def RotationMatrixToEulerAngles(R):
    """common/math.h:107-127 (host-side 3x3 math; the reference runs it once per frame)."""
    R = np.asarray(R, dtype=np.float64)
    sy = np.sqrt(R[0, 0] * R[0, 0] + R[1, 0] * R[1, 0])
    if not sy < 1e-6:
        return np.array([np.arctan2(R[2, 1], R[2, 2]), np.arctan2(-R[2, 0], sy), np.arctan2(R[1, 0], R[0, 0])])
    return np.array([np.arctan2(-R[1, 2], R[1, 1]), np.arctan2(-R[2, 0], sy), 0.0])


def AverageTransforms(transforms):
    """common::AverageTransforms (common/math.cc:177-195): mean translation, mean Euler angles
    (yaw * pitch * roll composition).  Used by the front end between Align and the second
    MotionCompensation when motion_compensation_options.use_average is set
    (map_builder.cc:333-341)."""
    ts = [np.asarray(t, dtype=np.float64) for t in transforms]
    if not ts:
        raise CheckFailure("Check failed: !transforms.empty() (common/math.cc:180)")
    tr = sum(t[:3, 3] for t in ts) / float(len(ts))
    ang = sum(RotationMatrixToEulerAngles(t[:3, :3]) for t in ts) / float(len(ts))

    def quat(angle, axis):
        q = np.zeros(4)
        q[0] = np.cos(0.5 * angle)
        q[1 + axis] = np.sin(0.5 * angle)
        return q

    def mul(a, b):
        return np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3],
                         a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                         a[0] * b[2] + a[2] * b[0] + a[3] * b[1] - a[1] * b[3],
                         a[0] * b[3] + a[3] * b[0] + a[1] * b[2] - a[2] * b[1]])

    w, x, y, z = mul(mul(quat(ang[2], 2), quat(ang[1], 1)), quat(ang[0], 0))
    tx, ty, tz = 2.0 * x, 2.0 * y, 2.0 * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz = tx * x, ty * x, tz * x
    tyy, tyz, tzz = ty * y, tz * y, tz * z
    out = np.eye(4)
    out[:3, :3] = [[1.0 - (tyy + tzz), txy - twz, txz + twy],
                   [txy + twz, 1.0 - (txx + tzz), tyz - twx],
                   [txz - twy, tyz + twx, 1.0 - (txx + tyy)]]
    out[:3, 3] = tr
    return out


def VoxelGridFilter(cloud, voxel_size, device=0):
    """pre_processers::filter::VoxelGrid::Filter (pre_processors/filter_voxel_grid.cc:37-78) on
    the GPU.  `cloud`: (N,5) float32 InnerPointType rows; returns the (M,5) voxel means in
    ascending (ix, iy, iz) order (the reference's order is std::unordered_map iteration order)."""
    lib = _lib.lib()
    pts = np.ascontiguousarray(np.asarray(cloud, dtype=np.float32))
    if pts.ndim != 2 or pts.shape[1] != 5:
        raise ValueError("cloud must be (N,5): x, y, z, intensity, factor")
    out = np.empty_like(pts)
    m = C.c_int64(0)
    rc = lib.sm_voxel_grid_filter(device, pts.ctypes.data, pts.shape[0], 20, float(voxel_size), out.ctypes.data,
                                  C.byref(m))
    if rc == -20:
        raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
    if rc == -1:
        raise CheckFailure("VoxelGrid: invalid voxel_size (ConfigsValid) or a coordinate outside the voxel index range")
    if rc != 0:
        raise RuntimeError(f"sm_voxel_grid_filter failed with {rc}")
    return out[:m.value].copy()


class M2dp:
    """descriptor::M2dp (descriptor/m2dp.h:45-84) on the GPU: setInputCloud / getFinalDescriptor."""

    def __init__(self, r=0.1, max_distance=100.0, t=16, p=4, q=16, device=0):
        self.r, self.max_distance, self.t, self.p, self.q, self.device = float(r), float(max_distance), int(t), int(p), int(q), device
        self._descriptor = None
        self.signature_matrix = None

    def setInputCloud(self, cloud):
        """cloud: InnerCloud or (N,3)/(N,5) float32 array.  Returns False for an empty cloud (m2dp.cc:130-133)."""
        pts = cloud.points if isinstance(cloud, InnerCloud) else np.ascontiguousarray(np.asarray(cloud, dtype=np.float32))
        lib = _lib.lib()
        n = lib.sm_m2dp_descriptor_length(self.r, self.max_distance, self.t, self.p, self.q)
        if n < 0:
            raise CheckFailure("M2dp: r is too small (m2dp.cc:64-67) or bad parameters")
        desc = np.zeros(n, np.float32)
        A = np.zeros((self.p * self.q, (n - self.p * self.q)), np.int32)
        rc = lib.sm_m2dp(self.device, pts.ctypes.data, pts.shape[0], 4 * pts.shape[1], self.r, self.max_distance,
                         self.t, self.p, self.q, desc.ctypes.data, n, A.ctypes.data)
        if rc == -20:
            raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
        if rc < 0:
            raise CheckFailure(f"sm_m2dp failed with {rc}")
        if rc == 0:
            return False
        self._descriptor, self.signature_matrix = desc, A
        return True

    def getFinalDescriptor(self):
        return self._descriptor


def matchTwoM2dpDescriptors(P, Q):
    """descriptor::matchTwoM2dpDescriptors (m2dp.cc:155-170): |Pearson correlation| in (0, 1), -1 on mismatch."""
    P = np.ascontiguousarray(P, np.float32); Q = np.ascontiguousarray(Q, np.float32)
    if P.shape != Q.shape:
        return -1.0
    return float(_lib.lib().sm_m2dp_match(P.ctypes.data, Q.ctypes.data, P.shape[0]))


class MrvmSettings(C.Structure):
    """MrvmSettings (builder/multi_resolution_voxel_map.h:55-66) == sm_mrvm_settings; the reference's defaults."""
    _fields_ = [("output_average", C.c_int32), ("output_rgb", C.c_int32), ("use_max_intensity", C.c_int32),
                ("prob_threshold", C.c_float), ("low_resolution", C.c_float), ("high_resolution", C.c_float),
                ("hit_prob", C.c_float), ("miss_prob", C.c_float), ("z_offset", C.c_float),
                ("max_point_num_in_cell", C.c_int32)]

    def __init__(self, output_average=False, output_rgb=False, use_max_intensity=True, prob_threshold=0.6,
                 low_resolution=1.0, high_resolution=0.1, hit_prob=0.55, miss_prob=0.48, z_offset=0.0,
                 max_point_num_in_cell=10):
        super().__init__(int(output_average), int(output_rgb), int(use_max_intensity), prob_threshold, low_resolution,
                         high_resolution, hit_prob, miss_prob, z_offset, int(max_point_num_in_cell))


class MultiResolutionVoxelMap:
    """builder::MultiResolutionVoxelMap (multi_resolution_voxel_map.{h,cc}) on the GPU: the ray-casting occupancy
    map that removes moving objects from static_map.pcd.  The map stays on the device between inserts.  Semantics:
    the reference's run by one thread; voxels are output in ascending (ix, iy, iz) order (include/sm_b200.h)."""

    def __init__(self, device=0, expected_voxels=1 << 20):
        self.device, self.expected_voxels = device, int(expected_voxels)
        self.settings = None
        self._h = None

    def __del__(self):
        self._release()

    def _release(self):
        if getattr(self, "_h", None):
            _lib.lib().sm_mrvm_destroy(self._h)
            self._h = None

    def _check(self, rc, what):
        if rc == -20:
            raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
        if rc == -1:
            raise CheckFailure(f"MultiResolutionVoxelMap::{what}: invalid argument")
        if rc < 0:
            raise RuntimeError(f"MultiResolutionVoxelMap::{what} failed with {rc}")
        return rc

    def Initialise(self, settings: MrvmSettings):
        """Initialise (:42-48) on an empty map.  CheckFailure where map_builder_options.cc:66-68 CHECK-fails
        (hit_prob <= 0.5, miss_prob >= 0.5, max_point_num_in_cell < 1) or high_resolution <= 0."""
        self._release()
        h = C.c_void_p()
        self._check(_lib.lib().sm_mrvm_create(self.device, C.byref(settings), self.expected_voxels, C.byref(h)),
                    "Initialise")
        self._h, self.settings = h, settings

    def SetOffsetZ(self, offset):
        self._check(_lib.lib().sm_mrvm_set_offset_z(self._handle(), float(offset)), "SetOffsetZ")

    def _handle(self):
        if not self._h:
            raise CheckFailure("MultiResolutionVoxelMap: Initialise first")
        return self._h

    def InsertPointCloud(self, cloud, origin):
        """cloud: (N,5) float32 InnerPointType rows (x, y, z, intensity, factor) as a numpy array, or a C-contiguous
        float32 CUDA tensor of the same shape (read in place, after the work queued on torch's current stream).
        origin: sensor position (3,).  Returns the number of points dropped for a non-finite coordinate; raises
        CheckFailure (map unchanged) for a voxel index outside [-2^20, 2^20)."""
        o = np.ascontiguousarray(np.asarray(origin, dtype=np.float32).reshape(3))
        lib = _lib.lib()
        if hasattr(cloud, "is_cuda") and cloud.is_cuda:
            import torch
            if cloud.dtype != torch.float32 or cloud.dim() != 2 or cloud.shape[1] != 5 or not cloud.is_contiguous():
                raise ValueError("cloud must be a contiguous (N,5) float32 tensor")
            stream = torch.cuda.current_stream(cloud.device).cuda_stream
            rc = lib.sm_mrvm_insert_device(self._handle(), cloud.data_ptr(), cloud.shape[0], 20, o.ctypes.data, stream)
        else:
            pts = np.ascontiguousarray(np.asarray(cloud, dtype=np.float32))
            if pts.ndim != 2 or pts.shape[1] != 5:
                raise ValueError("cloud must be (N,5): x, y, z, intensity, factor")
            rc = lib.sm_mrvm_insert(self._handle(), pts.ctypes.data, pts.shape[0], 20, o.ctypes.data)
        return self._check(rc, "InsertPointCloud")

    def size(self):
        return int(_lib.lib().sm_mrvm_size(self._handle()))

    def OutputToPointCloud(self, threshold=None, rgb=None):
        """OutputToPointCloud (:125-215) -> (M,4) float32 {x, y, z, value}.  threshold defaults to
        settings.prob_threshold, rgb to settings.output_rgb; value is the intensity (PointXYZI) or the grey level
        (PointXYZRGB)."""
        h = self._handle()
        t = float(self.settings.prob_threshold if threshold is None else threshold)
        r = int(bool(self.settings.output_rgb if rgb is None else rgb))
        lib = _lib.lib()
        m = C.c_int64(0)
        rc = lib.sm_mrvm_output(h, t, r, None, 0, C.byref(m))
        if rc == -1 and m.value > 0:
            out = np.empty((m.value, 4), np.float32)
            rc = lib.sm_mrvm_output(h, t, r, out.ctypes.data, m.value, C.byref(m))
            self._check(rc, "OutputToPointCloud")
            return out
        self._check(rc, "OutputToPointCloud")
        return np.zeros((0, 4), np.float32)

    def PhaseMs(self):
        """Cumulative device time of the insert phases (CUDA events): upload, keys + sort + segments, table insert,
        rays, voxel update; and the number of inserts."""
        ms = np.zeros(6, np.float32)
        self._check(_lib.lib().sm_mrvm_phase_ms(self._handle(), ms.ctypes.data), "PhaseMs")
        return {"upload": float(ms[0]), "keys_sort_segments": float(ms[1]), "table_insert": float(ms[2]),
                "rays": float(ms[3]), "update": float(ms[4]), "inserts": int(ms[5])}

    def State(self):
        """Test hook sm_debug_mrvm_state: dict(keys, prob, max_intensity, npts, points (n, max_point_num_in_cell, 4))
        in ascending key order."""
        h = self._handle()
        n = self.size()
        mp = self.settings.max_point_num_in_cell
        keys = np.zeros(n, np.int64); prob = np.zeros(n, np.uint8)
        mi = np.zeros(n, np.int32); npts = np.zeros(n, np.int32); pts = np.zeros((n, mp, 4), np.float32)
        got = C.c_int64(0)
        self._check(_lib.lib().sm_debug_mrvm_state(h, keys.ctypes.data, prob.ctypes.data, mi.ctypes.data,
                                                   npts.ctypes.data, pts.ctypes.data, n, C.byref(got)), "State")
        return {"keys": keys, "prob": prob, "max_intensity": mi, "npts": npts, "points": pts}


class FilterChain:
    """sm_filter_chain_* (include/sm_b200.h): the stages of a pre_processers::filter::Factory on the GPU.  Thin: the
    Python filter classes below drive it, or any object with the same methods (the tests' serial oracle)."""

    def __init__(self, device=0):
        self.device = device
        h = C.c_void_p()
        rc = _lib.lib().sm_filter_chain_create(device, C.byref(h))
        if rc == -20:
            raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
        if rc < 0:
            raise RuntimeError(f"sm_filter_chain_create failed with {rc}")
        self._h = h

    def __del__(self):
        if getattr(self, "_h", None):
            _lib.lib().sm_filter_chain_destroy(self._h)
            self._h = None

    def add(self, name):
        return _lib.lib().sm_filter_chain_add(self._h, name.encode())

    def set_param(self, stage, name, type_, text):
        return _lib.lib().sm_filter_chain_set_param(self._h, stage, name.encode(), type_, text.encode())

    def valid(self, stage):
        return _lib.lib().sm_filter_chain_valid(self._h, stage)

    def set_seed(self, seed):
        return _lib.lib().sm_filter_chain_set_seed(self._h, int(seed) & ((1 << 64) - 1))

    def filter(self, points5):
        """(N,5) float32 -> (rc, (M,5) float32 records, (M,) int32 chain-input indices)."""
        p = np.ascontiguousarray(points5, np.float32)
        n = p.shape[0]
        out = np.empty((max(n, 1), 5), np.float32)
        kept = np.empty(max(n, 1), np.int32)
        m = C.c_int64(0)
        rc = _lib.lib().sm_filter_chain_filter(self._h, p.ctypes.data, n, 20, out.ctypes.data, n, C.byref(m),
                                               kept.ctypes.data)
        if rc == -1 and m.value > n:                   # VoxelGrid never grows a cloud; kept for completeness
            out = np.empty((m.value, 5), np.float32); kept = np.empty(m.value, np.int32)
            rc = _lib.lib().sm_filter_chain_filter(self._h, p.ctypes.data, n, 20, out.ctypes.data, m.value,
                                                   C.byref(m), kept.ctypes.data)
        return rc, out[:m.value].copy(), kept[:m.value].copy()

    def filter_device(self, cloud):
        """contiguous (N,5) float32 CUDA tensor -> (rc, (M,5) tensor, (M,) int32 tensor), on torch's current stream."""
        import torch
        if cloud.dtype != torch.float32 or cloud.dim() != 2 or cloud.shape[1] != 5 or not cloud.is_contiguous():
            raise ValueError("cloud must be a contiguous (N,5) float32 tensor")
        n = cloud.shape[0]
        out = torch.empty((max(n, 1), 5), dtype=torch.float32, device=cloud.device)
        kept = torch.empty(max(n, 1), dtype=torch.int32, device=cloud.device)
        m = C.c_int64(0)
        stream = torch.cuda.current_stream(cloud.device).cuda_stream
        rc = _lib.lib().sm_filter_chain_filter_device(self._h, cloud.data_ptr(), n, 20, out.data_ptr(), n,
                                                      C.byref(m), kept.data_ptr(), stream)
        return rc, out[:m.value], kept[:m.value]

    def stage_counts(self):
        ns = _lib.lib().sm_filter_chain_stage_counts(self._h, None, 0)
        c = np.zeros(max(ns, 1), np.int64)
        _lib.lib().sm_filter_chain_stage_counts(self._h, c.ctypes.data, ns)
        return c[:ns]

    def stage_ms(self):
        ns = _lib.lib().sm_filter_chain_stage_ms(self._h, None, 0)
        c = np.zeros(max(ns, 1), np.float32)
        _lib.lib().sm_filter_chain_stage_ms(self._h, c.ctypes.data, ns)
        return c[:ns]


def _records(cloud):
    """InnerCloud / (N,3) / (N,5) -> (N,5) float32 InnerPointType rows (intensity and factor 0 for xyz input)."""
    p = cloud.points if isinstance(cloud, InnerCloud) else np.asarray(cloud, np.float32)
    p = np.asarray(p, np.float32)
    if p.ndim != 2 or p.shape[1] not in (3, 5):
        raise ValueError("cloud must be (N,3) or (N,5) float32")
    if p.shape[1] == 3:
        p = np.concatenate([p, np.zeros((p.shape[0], 2), np.float32)], axis=1)
    return np.ascontiguousarray(p)


def _filter_check(rc, what):
    if rc == -20:
        raise RuntimeError("staticmapping_b200: no CUDA device (no CPU fallback)")
    if rc in (-1, -10, -11):
        raise CheckFailure(f"{what} failed with {rc}")
    if rc < 0:
        raise RuntimeError(f"{what} failed with {rc}")
    return rc


def _init_stage(chain, stage, name, node):
    """Interface::InitFromXmlNode (filter_interface.cc:29-60) on one stage -> ConfigsValid()."""
    if node.tag != "filter":
        raise CheckFailure(f"expected a <filter> node, got <{node.tag}>")
    if node.get("name", "") != name:
        return False
    for p in node.findall("param"):
        t = p.get("type")
        rc = chain.set_param(stage, p.get("name", ""), int(t) if t is not None else 2, p.text or "")
        if rc < 0:
            raise CheckFailure(f"{name}: param {p.get('name')!r} (type {t}) rejected with {rc}")
    return bool(chain.valid(stage))


class FilterFactory:
    """pre_processers::filter::Factory (filter_factory.cc:63-123) on the GPU: the <filters> chain of the XML config.
    `chain` replaces the GPU backend (tests pass the serial oracle).  Unknown filter names raise CheckFailure (the
    reference skips them), unknown parameters too (the reference CHECK-fails)."""

    def __init__(self, device=0, seed=0, chain=None):
        self._chain = chain if chain is not None else FilterChain(device)
        self._chain.set_seed(seed)
        self.names = []
        self._cloud = None

    def InitFromXmlText(self, text):
        self.InitFromXmlNode(ET.fromstring(text))

    def InitFromXmlNode(self, filters_node):
        for node in filters_node.findall("filter"):
            name = node.get("name", "")
            stage = self._chain.add(name)
            if stage < 0:
                raise CheckFailure(f"filter {name!r} is not supported ({stage})")
            _init_stage(self._chain, stage, name, node)
            self.names.append(name)

    def SetInputCloud(self, cloud):
        self._cloud = _records(cloud)

    def Filter(self):
        """-> (M,5) float32 records of the filtered cloud.  KeptIndex() gives their chain-input indices."""
        if self._cloud is None:
            raise CheckFailure("FilterFactory: SetInputCloud first")
        rc, out, kept = self._chain.filter(self._cloud)
        _filter_check(rc, "FilterFactory::Filter")
        self._kept = kept
        return out

    def FilterDevice(self, cloud):
        """contiguous (N,5) float32 CUDA tensor -> ((M,5) tensor, (M,) int32 chain-input indices); the cloud never
        leaves the device."""
        rc, out, kept = self._chain.filter_device(cloud)
        _filter_check(rc, "FilterFactory::FilterDevice")
        return out, kept

    def KeptIndex(self):
        return self._kept

    def StageCounts(self):
        return self._chain.stage_counts()

    def StageMs(self):
        return self._chain.stage_ms()


class _Filter:
    """One pre_processers::filter::Interface (filter_interface.h) on the GPU: a one-stage chain."""
    NAME = ""

    def __init__(self, device=0, seed=0, chain=None):
        self._chain = chain if chain is not None else FilterChain(device)
        self._chain.set_seed(seed)
        self._stage = _filter_check(self._chain.add(self.NAME), f"{self.NAME}()")
        self._cloud = None
        self._inliers = np.zeros(0, np.int64)
        self._outliers = np.zeros(0, np.int64)

    def InitFromXmlNode(self, node):
        return _init_stage(self._chain, self._stage, self.NAME, node)

    def InitFromXmlText(self, text):
        return self.InitFromXmlNode(ET.fromstring(text))

    def ConfigsValid(self):
        return bool(self._chain.valid(self._stage))

    def SetInputCloud(self, cloud):
        self._cloud = _records(cloud)
        self._inliers = np.zeros(0, np.int64)
        self._outliers = np.zeros(0, np.int64)

    def Filter(self):
        """-> (M,5) float32 records; Inliers() / Outliers() are updated like the reference's."""
        if self._cloud is None:
            raise CheckFailure(f"{self.NAME}: SetInputCloud first")
        rc, out, kept = self._chain.filter(self._cloud)
        _filter_check(rc, f"{self.NAME}::Filter")
        self._inliers = np.sort(kept[kept >= 0]).astype(np.int64)
        self._outliers = self._outlier_set()
        return out

    def _outlier_set(self):
        mask = np.ones(self._cloud.shape[0], bool)
        mask[self._inliers] = False
        return np.flatnonzero(mask).astype(np.int64)

    def Inliers(self):
        return self._inliers

    def Outliers(self):
        return self._outliers


class Range(_Filter):
    NAME = "Range"


class AxisRange(_Filter):
    NAME = "AxisRange"


class BoundingBoxRemoval(_Filter):
    NAME = "BoundingBoxRemoval"


class RandomSampler(_Filter):
    NAME = "RandomSampler"


class RangeImage(_Filter):
    NAME = "RangeImage"


class GroundRemoval2(_Filter):
    NAME = "GroundRemoval2"


class GroundRemoval(_Filter):
    NAME = "GroundRemoval"

    def __init__(self, device=0, seed=0, chain=None):
        super().__init__(device, seed, chain)
        self._leaf, self._min_pts = 0.8, 10

    def InitFromXmlNode(self, node):
        ok = super().InitFromXmlNode(node)
        for p in node.findall("param"):                 # the vanished voxels of Outliers() need these two
            if p.get("name") == "leaf_size":
                self._leaf = float(np.float32(float(p.text)) if p.get("type") == "1" else int(float(p.text)))
            if p.get("name") == "min_point_num_in_voxel":
                self._min_pts = int(float(p.text)) if p.get("type") == "1" else int(p.text)
        return ok

    def _outlier_set(self):
        """voxels below min_point_num_in_voxel vanish: their points are neither inliers nor outliers"""
        p = self._cloud[:, :3]
        fin = np.isfinite(p).all(axis=1)
        with np.errstate(invalid="ignore", over="ignore"):
            v = np.trunc(p / np.float32(self._leaf)).astype(np.int64)
        v[~fin] = 0
        _, inv, cnt = np.unique(v, axis=0, return_inverse=True, return_counts=True)
        small = (cnt[inv.reshape(-1)] < self._min_pts) & fin
        mask = ~small
        mask[self._inliers] = False
        return np.flatnonzero(mask).astype(np.int64)


class VoxelGrid(_Filter):
    """VoxelGrid::Filter: inliers and outliers stay empty, like the reference's (FilterPrepare clears them)."""
    NAME = "VoxelGrid"

    def Filter(self):
        out = super().Filter()
        self._inliers = self._outliers = np.zeros(0, np.int64)
        return out


class StatisticRemoval(_Filter):
    """StatisticRemoval: the identity; its body (and so its inliers / outliers) is commented out in the reference."""
    NAME = "StatisticRemoval"

    def Filter(self):
        out = super().Filter()
        self._inliers = self._outliers = np.zeros(0, np.int64)
        return out
