"""dataset.py -- host-side mirror of the reference's recorded-sequence reader and of the visual
odometry app's loop, feeding the CUDA solver.

Reference interfaces restated (names, argument meaning and behaviour kept; code is not shared):

* `CCameraRecord` (phovo/include/CCameraRecord.h:41-121): `SetFileName`, `Start` (throws if the record
  file cannot be opened, :63-72), `GetSensorData` (next non-comment line `timestamp filename`; the image
  path is relative to the record file's directory, :74-108; `None` when the file is exhausted), `Stop`.
  The image is decoded like `CImageReader` does (CImageReader.h:52-91): `cv::imread(file, 0)` for an
  8-bit intensity record (colour files are converted to grey by OpenCV), `cv::imread(file, -1)` for
  anything else (the 16-bit depth PNGs of the TUM RGB-D datasets stay raw).
* `CMultiSensorDataSource` (CMultiSensorDataSource.h:41-121): a map sensor id -> source; one
  `GetMultiSensorData()` call takes the NEXT item of every source (records are paired by ORDER, not by
  timestamp) and returns nothing as soon as one source is exhausted (:73-92).
* the loop of apps/PhotoconsistencyVisualOdometry/PhotoconsistencyVisualOdometry.cpp:196-262:
  previous frame = source, current frame = target, the SAME initial state every frame (:175, :224),
  `pose *= Rt^-1` (:234), quaternion of the rotation block, one line
  `timestamp tx ty tz qx qy qz qw` per frame with `setprecision(digits10 + 1)` (:240-243).

What is B200-specific: depth stays raw u16 on the host and is scaled by `depthScalingFactor` on the
device (`(double)raw * scale`, the same product the app forms in `Mat_<double> * scalar`, :208/:220);
`PrefetchingSource` decodes the PNGs on a pool of background threads into a ring of PINNED buffers (in
record order), so decode -- the slowest stage of a recorded sequence by two orders of magnitude -- runs
on several cores beside the alignment and every upload runs at full PCIe speed; frame k's target
pyramid is promoted to frame k+1's source pyramid on the device instead of being rebuilt.
"""
import os
import queue
import threading

import numpy as np

IntensityCameraIdentifier = "intensity_camera"      # CSensorIdentifier.h
DepthCameraIdentifier = "depth_camera"


class SensorData(object):
    """CSensorData: a time-stamped datum."""

    def __init__(self, time_stamp, data):
        self._t, self._d = time_stamp, data

    def GetTimeStamp(self):
        return self._t

    def GetData(self):
        return self._d


class CCameraRecord(object):
    """One `timestamp filename` record file of a recorded sequence (rgb.txt / depth.txt)."""

    def __init__(self, intensity):
        """intensity=True: 8-bit grey images (`imread(file, 0)`); False: unchanged (`imread(file, -1)`)."""
        self._intensity = bool(intensity)
        self._name = None
        self._fh = None

    def SetFileName(self, file_name):
        self._name = str(file_name)

    def Start(self):
        try:
            self._fh = open(self._name, "r")
        except (OSError, TypeError):
            raise RuntimeError("Unable to open camera record file %s" % self._name)

    def next_entry(self):
        """(timestamp, absolute image path) of the next record line, or None at the end of the file."""
        if self._fh is None:
            raise RuntimeError("camera record %s has not been started" % self._name)
        for line in self._fh:
            if not line.strip() or line[0] == "#":
                continue
            fields = line.split()
            if len(fields) < 2:
                continue
            return float(fields[0]), os.path.join(os.path.dirname(os.path.abspath(self._name)), fields[1])
        return None

    def read_image(self, path):
        import cv2
        img = cv2.imread(path, cv2.IMREAD_GRAYSCALE if self._intensity else cv2.IMREAD_UNCHANGED)
        if img is None:
            raise RuntimeError("Unable to read image %s" % path)
        return img

    def GetSensorData(self):
        e = self.next_entry()
        if e is None:
            return None
        return SensorData(e[0], self.read_image(e[1]))

    # CSensorDataSourceBase::GetData is what CMultiSensorDataSource calls
    GetData = GetSensorData

    def Stop(self):
        if self._fh is not None:
            self._fh.close()
            self._fh = None


class CMultiSensorDataSource(object):
    def __init__(self):
        self._sources = {}

    def SetSensorDataSource(self, sensor_id, source):
        self._sources.setdefault(sensor_id, source)       # std::map::insert keeps the first

    def Start(self):
        for k in sorted(self._sources):
            self._sources[k].Start()

    def GetMultiSensorData(self):
        out = {}
        for k in sorted(self._sources):                   # std::map order
            d = self._sources[k].GetData()
            if d is None:
                return None
            out[k] = d
        return out

    def Stop(self):
        for k in sorted(self._sources):
            self._sources[k].Stop()


def open_rgbd_dataset(directory):
    """The app's input convention (VisualOdometry.cpp:92-107): <dir>/rgb.txt and <dir>/depth.txt."""
    rgb, depth = os.path.join(directory, "rgb.txt"), os.path.join(directory, "depth.txt")
    for f in (rgb, depth):
        if not os.path.exists(f):
            raise RuntimeError("Input data file %s does not exist" % f)
    src = CMultiSensorDataSource()
    a, b = CCameraRecord(True), CCameraRecord(False)
    a.SetFileName(rgb)
    b.SetFileName(depth)
    src.SetSensorDataSource(IntensityCameraIdentifier, a)
    src.SetSensorDataSource(DepthCameraIdentifier, b)
    return src


class PrefetchingSource(object):
    """Runs a CMultiSensorDataSource ahead of its consumer on background threads.  PNG decoding is what
    bounds a recorded sequence (a 640x480 colour + 16-bit depth pair takes ~5-20 ms per core, the solver
    0.2 ms), so the frames are decoded by a pool of `workers` threads (cv2 releases the GIL) and handed
    over in record order.  Every decoded image is copied into a slot of a ring of page-locked host
    buffers (when CUDA is available), so that the solver's uploads are direct DMA.  A slot is recycled
    `ahead + workers + 3` frames later: up to `workers` frames are being decoded, `ahead` wait in the
    queue, one is in hand-over, and the consumer may hold the current and the previous frame.
    Iterating yields {sensor id: SensorData}; errors of the workers are re-raised in the consumer.
    Sources that are not CCameraRecord-like (no next_entry / read_image) are read sequentially."""

    def __init__(self, source, ahead=4, pin=None, workers=4):
        self._src, self._ahead, self._workers = source, max(1, int(ahead)), max(1, int(workers))
        self._q = queue.Queue(maxsize=self._ahead)
        self._ring, self._lock = {}, threading.Lock()
        if pin is None:
            try:
                import torch
                pin = torch.cuda.is_available()
            except Exception:
                pin = False
        self._pin = bool(pin)
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._work, daemon=True)

    def _buffer(self, key, like, slot):
        slots = self._ahead + self._workers + 3
        k = (key, like.shape, like.dtype.str)
        with self._lock:
            if k not in self._ring:
                if self._pin:
                    import torch
                    tdt = {"|u1": torch.uint8, "<u2": torch.int16, "<f4": torch.float32, "<f8": torch.float64}[like.dtype.str]
                    self._ring[k] = [torch.empty(like.shape, dtype=tdt).pin_memory().numpy().view(like.dtype) for _ in range(slots)]
                else:
                    self._ring[k] = [np.empty(like.shape, like.dtype) for _ in range(slots)]
            return self._ring[k][slot % slots]

    def _stage(self, item, slot):
        staged = {}
        for key, sd in item.items():
            buf = self._buffer(key, sd.GetData(), slot)
            np.copyto(buf, sd.GetData())
            staged[key] = SensorData(sd.GetTimeStamp(), buf)
        return staged

    def _records(self):
        """{id: record} if every source can be split into (next line, decode), else None."""
        srcs = getattr(self._src, "_sources", None)
        if not srcs or not all(hasattr(r, "next_entry") and hasattr(r, "read_image") for r in srcs.values()):
            return None
        return srcs

    def _put(self, item):
        while not self._stop.is_set():
            try:
                self._q.put(item, timeout=0.1)
                return
            except queue.Full:
                pass

    def _work(self):
        try:
            self._src.Start()
            records = self._records()
            slot = 0
            if records is None or self._workers == 1:
                while not self._stop.is_set():
                    item = self._src.GetMultiSensorData()
                    if item is None:
                        break
                    self._put(self._stage(item, slot))
                    slot += 1
            else:
                import collections
                from concurrent.futures import ThreadPoolExecutor

                def decode(entries, slot_):
                    return self._stage({k: SensorData(ts, records[k].read_image(path)) for k, (ts, path) in entries.items()}, slot_)

                pending, exhausted = collections.deque(), False
                with ThreadPoolExecutor(self._workers) as pool:
                    while not self._stop.is_set():
                        while not exhausted and len(pending) < self._workers:
                            entries = {}
                            for k in sorted(records):              # one line of every record, like GetMultiSensorData
                                e = records[k].next_entry()
                                if e is None:
                                    exhausted = True
                                    break
                                entries[k] = e
                            if exhausted:
                                break
                            pending.append(pool.submit(decode, entries, slot))
                            slot += 1
                        if not pending:
                            break
                        self._put(pending.popleft().result())
                    for f in pending:
                        f.cancel()
            self._src.Stop()
            self._q.put(None)
        except Exception as e:      # noqa: BLE001 -- handed to the consumer
            self._q.put(e)

    def __iter__(self):
        self._thread.start()
        try:
            while True:
                item = self._q.get()
                if item is None:
                    return
                if isinstance(item, Exception):
                    raise item
                yield item
        finally:
            self._stop.set()


def quaternion_of(R):
    """(x, y, z, w) of a rotation matrix with the branches of Eigen::Quaternion(Matrix3) (VisualOdometry.cpp:237)."""
    R = np.asarray(R, dtype=np.float64)
    q = np.zeros(4)
    t = R[0, 0] + R[1, 1] + R[2, 2]
    if t > 0:
        t = np.sqrt(t + 1.0)
        q[3] = 0.5 * t
        t = 0.5 / t
        q[0], q[1], q[2] = (R[2, 1] - R[1, 2]) * t, (R[0, 2] - R[2, 0]) * t, (R[1, 0] - R[0, 1]) * t
    else:
        i = 0
        if R[1, 1] > R[0, 0]:
            i = 1
        if R[2, 2] > R[i, i]:
            i = 2
        j, k = (i + 1) % 3, (i + 2) % 3
        t = np.sqrt(R[i, i] - R[j, j] - R[k, k] + 1.0)
        q[i] = 0.5 * t
        t = 0.5 / t
        q[3] = (R[k, j] - R[j, k]) * t
        q[j] = (R[j, i] + R[i, j]) * t
        q[k] = (R[k, i] + R[i, k]) * t
    return q


def trajectory_line(time_stamp, pose):
    """`timestamp tx ty tz qx qy qz qw`, 16 significant digits like setprecision(digits10 + 1) (:240-243)."""
    q = quaternion_of(pose[:3, :3])
    return " ".join("%.16g" % v for v in (time_stamp, pose[0, 3], pose[1, 3], pose[2, 3], q[0], q[1], q[2], q[3]))


def run_visual_odometry(odometry, source, trajectory_file=None, depth_scaling_factor=1. / 5000.,
                        initial_state=None, promote=True, on_frame=None):
    """The loop of PhotoconsistencyVisualOdometry.cpp:196-262 over `source` (a CMultiSensorDataSource, a
    PrefetchingSource or any iterable of {id: SensorData}).  `odometry` is a configured
    CPhotoconsistencyOdometryCuda (SetConfig / ReadConfigurationFile + SetIntrinsicMatrix done).
    Depth images of an integer type are uploaded raw and scaled on the device, float images are
    multiplied here as the app does.  Returns [(timestamp, pose 4x4)] for frames 1..N-1; writes the TUM
    trajectory if `trajectory_file` is given.  `on_frame(k, item, Rt)` is called after every alignment
    (the apps' warpImage / absdiff display goes there)."""
    if isinstance(source, CMultiSensorDataSource):
        def frames():
            source.Start()
            try:
                while True:
                    item = source.GetMultiSensorData()
                    if item is None:
                        return
                    yield item
            finally:
                source.Stop()
        it = frames()
    else:
        it = iter(source)
    state0 = np.zeros(6) if initial_state is None else np.asarray(initial_state, dtype=np.float64)

    def depth_of(item):
        d = item[DepthCameraIdentifier].GetData()
        if d.dtype.kind in "ui":
            return d if d.dtype == np.uint16 else d.astype(np.uint16), depth_scaling_factor
        return np.asarray(d, dtype=np.float64) * depth_scaling_factor, 1.0

    out = open(trajectory_file, "w") if trajectory_file else None
    poses = []
    try:
        prev = next(it, None)
        if prev is None:
            return poses
        pose = np.eye(4)
        k = 0
        prev_depth = None
        for cur in it:
            k += 1
            d, s = depth_of(prev) if prev_depth is None else prev_depth
            if promote and k > 1:
                odometry.PromoteTargetToSource(d, depth_scale=s)          # frame k-1's target pyramid is frame k's source
            else:
                odometry.SetSourceFrame(prev[IntensityCameraIdentifier].GetData(), d, depth_scale=s)
            # the app passes the current depth too; only the photometric + depth solver reads it
            prev_depth = depth_of(cur)
            odometry.SetTargetFrame(cur[IntensityCameraIdentifier].GetData(), prev_depth[0], depth_scale=prev_depth[1])
            odometry.SetInitialStateVector(state0)
            odometry.Optimize()
            Rt = odometry.GetOptimalRigidTransformationMatrix()
            pose = pose @ np.linalg.inv(Rt)                                # :234
            ts = cur[IntensityCameraIdentifier].GetTimeStamp()
            poses.append((ts, pose.copy()))
            if out:
                out.write(trajectory_line(ts, pose) + "\n")
            if on_frame:
                on_frame(k, cur, Rt)
            prev = cur
    finally:
        if out:
            out.close()
    return poses
