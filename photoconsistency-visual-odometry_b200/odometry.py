"""Python mirror of the reference's solver interface over the C ABI.

`CPhotoconsistencyOdometryCuda` has the same methods, argument meaning and call order as
`phovo::CPhotoconsistencyOdometry<TPixel,TCoordinate>` (CPhotoconsistencyOdometry.h:137-179) and
its analytic implementation (CPhotoconsistencyOdometryAnalytic.h:448-607), so tests read like
the reference apps (PhotoconsistencyFrameAlignment.cpp:90-105).  The C++ adapter with the
identical surface is include/CPhotoconsistencyOdometryCuda.h.  All compute happens in
libphovo_b200.so on the GPU; nothing here has a CPU path.
"""
import ctypes as C
import os

import numpy as np

from . import capi
from .capi import PhovoError


class CPhotoconsistencyOdometryCuda:
    def __init__(self, device=0, mode=capi.MODE_ANALYTIC_REF):
        self._L = capi.lib()
        h = C.c_void_p()
        rc = self._L.phovo_create(device, C.byref(h))
        if rc != capi.OK:
            raise PhovoError(rc, (self._L.phovo_last_error(None) or b"").decode())
        self._h = h
        self._check(self._L.phovo_set_mode(self._h, mode))

    # -- plumbing -------------------------------------------------------------------------
    def _check(self, rc):
        if rc != capi.OK:
            raise PhovoError(rc, (self._L.phovo_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.phovo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference interface --------------------------------------------------------------
    def ReadConfigurationFile(self, fileName):                      # AN:581-607 / CE:526-576
        self._check(self._L.phovo_load_config_yaml(self._h, os.fsencode(fileName)))

    def SetMinDepth(self, minD):                                    # AN:448-451
        cfg = self.GetConfig()
        self._check(self._L.phovo_set_depth_range(self._h, float(minD), cfg.max_depth))

    def SetMaxDepth(self, maxD):                                    # AN:454-457
        cfg = self.GetConfig()
        self._check(self._L.phovo_set_depth_range(self._h, cfg.min_depth, float(maxD)))

    def SetIntrinsicMatrix(self, intrinsicMatrix):                  # AN:460-463
        K = np.ascontiguousarray(intrinsicMatrix, dtype=np.float64).reshape(9)
        self._check(self._L.phovo_set_intrinsics(self._h, K.ctypes.data_as(capi._dp)))
        self._K = K.reshape(3, 3).copy()

    def _follow_producer_stream(self, *images):
        """A CUDA tensor is produced on torch's current stream of its device: run the context on that
        stream, so that the library's kernels are ordered after the producer (the C ABI reads device
        pointers in place on the context's stream, include/phovo_b200.h: phovo_set_source)."""
        for img in images:
            if img is None or isinstance(img, np.ndarray) or not getattr(img, "is_cuda", False):
                continue
            import torch
            stream = torch.cuda.current_stream(img.device).cuda_stream
            if getattr(self, "_bound_stream", None) != stream:
                self.SetStream(stream)
            return

    @staticmethod
    def _depth_args(depthImage, depth_scale):
        if isinstance(depthImage, np.ndarray):
            if depthImage.dtype == np.float64:
                t = capi.DEPTH_F64
            elif depthImage.dtype == np.float32:
                t = capi.DEPTH_F32
            elif depthImage.dtype == np.uint16:
                t = capi.DEPTH_U16
            else:
                raise TypeError("depth must be float64, float32 or uint16")
            if depthImage.strides[1] != depthImage.itemsize:
                depthImage = np.ascontiguousarray(depthImage)
            return depthImage, t, depthImage.strides[0], depthImage.ctypes.data
        # torch tensor (host pinned or device)
        import torch
        t = {torch.float64: capi.DEPTH_F64, torch.float32: capi.DEPTH_F32, torch.uint16: capi.DEPTH_U16,
             torch.int16: capi.DEPTH_U16}[depthImage.dtype]
        return depthImage, t, depthImage.stride(0) * depthImage.element_size(), depthImage.data_ptr()

    @staticmethod
    def _gray_args(img):
        if isinstance(img, np.ndarray):
            if img.dtype != np.uint8:
                raise TypeError("intensity image must be uint8")
            if img.strides[1] != 1:
                img = np.ascontiguousarray(img)
            return img, img.strides[0], img.ctypes.data, img.shape
        return img, img.stride(0), img.data_ptr(), tuple(img.shape)

    def SetSourceFrame(self, intensityImage, depthImage, depth_scale=1.0):   # AN:466-476
        self._follow_producer_stream(intensityImage, depthImage)
        g, gstep, gptr, shape = self._gray_args(intensityImage)
        d, dtype, dstep, dptr = self._depth_args(depthImage, depth_scale)
        if tuple(d.shape) != tuple(shape):
            raise ValueError("intensity and depth image sizes differ")
        self._check(self._L.phovo_set_source(self._h, gptr, gstep, dptr, dtype, dstep, float(depth_scale),
                                             shape[0], shape[1]))

    def SetTargetFrame(self, intensityImage, depthImage=None, depth_scale=1.0):
        """AN:479-491: the analytic and Ceres solvers ignore the target depth (AN:484); the photometric +
        depth solver (MODE_BIOBJECTIVE, BiObjective.h:567-579) needs it."""
        self._follow_producer_stream(intensityImage, depthImage)
        g, gstep, gptr, shape = self._gray_args(intensityImage)
        self._check(self._L.phovo_set_target(self._h, gptr, gstep, shape[0], shape[1]))
        if depthImage is not None and self.GetConfig().mode == capi.MODE_BIOBJECTIVE:
            d, dtype, dstep, dptr = self._depth_args(depthImage, depth_scale)
            self._check(self._L.phovo_set_target_depth(self._h, dptr, dtype, dstep, float(depth_scale)))

    def SetInitialStateVector(self, initialStateVector):            # AN:494-497
        s = np.ascontiguousarray(initialStateVector, dtype=np.float64).reshape(6)
        self._check(self._L.phovo_set_initial_state(self._h, s.ctypes.data_as(capi._dp)))

    def Optimize(self):                                             # AN:500-563
        self._check(self._L.phovo_optimize(self._h))

    def GetOptimalStateVector(self):                                # AN:566-569
        s = np.zeros(6)
        self._check(self._L.phovo_get_state(self._h, s.ctypes.data_as(capi._dp)))
        return s

    def GetOptimalRigidTransformationMatrix(self):                  # AN:572-578
        m = np.zeros(16)
        self._check(self._L.phovo_get_rt(self._h, m.ctypes.data_as(capi._dp)))
        return m.reshape(4, 4)

    # -- diagnostics of the apps (phovo::warpImage, CPhotoconsistencyOdometry.h:73-134) ------
    def WarpImage(self, intensityImage, depthImage, Rt, intrinsicMatrix, level=0, targetImage=None, depth_scale=1.0):
        """Returns the warped source image (u8); with `targetImage` also |target - warped| as the
        apps display it (FrameAlignment.cpp:107-110).  numpy inputs."""
        g, gstep, gptr, shape = self._gray_args(np.ascontiguousarray(intensityImage))
        d, dtype, dstep, dptr = self._depth_args(np.ascontiguousarray(depthImage), depth_scale)
        rt = np.ascontiguousarray(Rt, dtype=np.float64).reshape(16)
        K = np.ascontiguousarray(intrinsicMatrix, dtype=np.float64).reshape(9)
        warped = np.zeros(shape, np.uint8)
        diff = tgt = None
        if targetImage is not None:
            tgt = np.ascontiguousarray(targetImage, dtype=np.uint8)
            diff = np.zeros(shape, np.uint8)
        self._check(self._L.phovo_warp_image(self._h, gptr, gstep, dptr, dtype, dstep, float(depth_scale), shape[0], shape[1],
                                             rt.ctypes.data_as(capi._dp), K.ctypes.data_as(capi._dp), int(level),
                                             warped.ctypes.data, warped.strides[0],
                                             None if tgt is None else tgt.ctypes.data, 0 if tgt is None else tgt.strides[0],
                                             None if diff is None else diff.ctypes.data, 0 if diff is None else diff.strides[0]))
        return warped if diff is None else (warped, diff)

    # -- extensions (not in the reference) --------------------------------------------------
    def SetConfig(self, cfg):
        self._check(self._L.phovo_set_config(self._h, C.byref(cfg)))

    def GetConfig(self):
        cfg = capi.Config()
        self._check(self._L.phovo_get_config(self._h, C.byref(cfg)))
        return cfg

    def SetMode(self, mode):
        self._check(self._L.phovo_set_mode(self._h, mode))

    def SetUseGraph(self, enable):
        self._check(self._L.phovo_set_use_graph(self._h, int(enable)))

    def SetBuildAllLevels(self, enable):
        self._check(self._L.phovo_set_build_all_levels(self._h, int(enable)))

    def SetStream(self, cuda_stream):
        self._check(self._L.phovo_set_stream(self._h, cuda_stream))
        self._bound_stream = cuda_stream

    def SetExecution(self, path):
        """2 persistent cooperative kernel per level (default), 3 the same with small levels inside one
        thread-block cluster, 1 CUDA graph, 0 stream launches."""
        self._check(self._L.phovo_set_execution(self._h, int(path)))

    def LastPath(self):
        return int(self._L.phovo_last_optimize_path(self._h))

    def UsedGraph(self):
        return bool(self._L.phovo_last_optimize_used_graph(self._h))

    def GraphError(self):
        return (self._L.phovo_graph_error(self._h) or b"").decode()

    def PromoteTargetToSource(self, depthImage, depth_scale=1.0):
        self._follow_producer_stream(depthImage)
        d, dtype, dstep, dptr = self._depth_args(depthImage, depth_scale)
        self._check(self._L.phovo_promote_target_to_source(self._h, dptr, dtype, dstep, float(depth_scale)))

    def IterationStats(self):
        out = []
        for i in range(self._L.phovo_num_iter_stats(self._h)):
            s = capi.IterStats()
            self._check(self._L.phovo_get_iter_stats(self._h, i, C.byref(s)))
            out.append(s.as_dict())
        return out

    def LevelImage(self, which, level):
        r, c = C.c_int32(), C.c_int32()
        self._check(self._L.phovo_get_level_image(self._h, which, level, None, C.byref(r), C.byref(c)))
        out = np.zeros((r.value, c.value), dtype=np.float64)
        self._check(self._L.phovo_get_level_image(self._h, which, level, out.ctypes.data, C.byref(r), C.byref(c)))
        return out

    def EvalNormalEquations(self, level, state):
        s = np.ascontiguousarray(state, dtype=np.float64).reshape(6)
        st = capi.IterStats()
        self._check(self._L.phovo_eval_normal_equations(self._h, level, s.ctypes.data_as(capi._dp), C.byref(st)))
        return st.as_dict()

    def EvalResiduals(self, level, state, shape=None):
        """Residual vector and Jacobian at `state` on `level`: rows*cols rows of that level, or 2*rows*cols in the
        photometric + depth mode, which stacks a depth row under every intensity row.  The buffers are sized from the
        level the context built; `shape`, if given, must be that level's (rows, cols)."""
        s = np.ascontiguousarray(state, dtype=np.float64).reshape(6)
        r, c = C.c_int32(), C.c_int32()
        self._check(self._L.phovo_get_level_image(self._h, 0, level, None, C.byref(r), C.byref(c)))
        if shape is not None and tuple(shape) != (r.value, c.value):
            raise ValueError("level %d is %dx%d, not %s" % (level, r.value, c.value, tuple(shape)))
        n = r.value * c.value * (2 if self.GetConfig().mode == capi.MODE_BIOBJECTIVE else 1)
        res, jac = np.zeros(n), np.zeros((n, 6))
        self._check(self._L.phovo_eval_residuals(self._h, level, s.ctypes.data_as(capi._dp), res.ctypes.data, jac.ctypes.data))
        return res, jac

    def Timings(self):
        a, b = C.c_float(), C.c_float()
        self._check(self._L.phovo_get_timings(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def LaunchCount(self):
        return int(self._L.phovo_launch_count(self._h))

    def Synchronize(self):
        self._check(self._L.phovo_synchronize(self._h))

    # batch of independent pairs --------------------------------------------------------------
    def BatchLastPath(self):
        """1: the shared-memory-resident batch kernels ran; 3: waves of per-pair slots, one CTA per pair through every level
        (Ceres / photometric + depth solver, blurred or large levels); 2: the pool of per-pair contexts (debug flag 4)."""
        return int(self._L.phovo_batch_last_path(self._h))

    def BatchAlign(self, gray0, depth0, gray1, initial_states=None, depth_scale=1.0, depth1=None):
        """Host (numpy / pinned torch) or device (torch) arrays [P,R,C]; returns (states[P,6], iterations[P,MAXL]).
        `depth1` (target depth, same type as depth0) is read by the photometric + depth solver only.  The library reads
        dense frames: strided views are copied first."""
        gray0, depth0, gray1, depth1 = (self._dense(a) for a in (gray0, depth0, gray1, depth1))
        self._follow_producer_stream(gray0, depth0, gray1, depth1)     # (device copies made above are on torch's stream)
        P, R, Cc = tuple(gray0.shape)
        dtype = self._batch_depth_type(depth0)
        if tuple(depth0.shape) != (P, R, Cc) or tuple(gray1.shape) != (P, R, Cc) or (depth1 is not None and tuple(depth1.shape) != (P, R, Cc)):
            raise ValueError("gray0, depth0, gray1 and depth1 must all be [P, rows, cols]")
        if depth1 is not None and self._batch_depth_type(depth1) != dtype:
            raise TypeError("depth1 must have the element type of depth0 (one depth type is passed for both)")
        states = np.zeros((P, 6))
        iters = np.zeros((P, capi.MAXL), dtype=np.int32)
        init = None if initial_states is None else np.ascontiguousarray(initial_states, dtype=np.float64)
        if init is not None and init.size != P * 6:
            raise ValueError("initial_states must be [P, 6]")
        if depth1 is not None:
            self._check(self._L.phovo_batch_align_with_target_depth(self._h, P, R, Cc, capi._ptr(gray0), capi._ptr(depth0), dtype,
                                                                    float(depth_scale), capi._ptr(gray1), capi._ptr(depth1), capi._ptr(init),
                                                                    states.ctypes.data, iters.ctypes.data))
            return states, iters
        self._check(self._L.phovo_batch_align(self._h, P, R, Cc, capi._ptr(gray0), capi._ptr(depth0), dtype,
                                              float(depth_scale), capi._ptr(gray1), capi._ptr(init),
                                              states.ctypes.data, iters.ctypes.data))
        return states, iters

    def BatchAlignDevice(self, gray0, depth0, gray1, states_out, iters_out, initial_states=None, depth_scale=1.0, depth1=None):
        """All torch device tensors; asynchronous on the context stream (torch's current stream of the
        tensors' device: inputs are ordered after their producers, outputs before their consumers).
        `depth1` (target depth, depth0's shape and element type) is read by the photometric + depth solver only; with it
        that solver's pairs go through the pool or the slot waves and the call returns once the outputs are written."""
        import torch
        if depth1 is not None:
            gray0, depth0, gray1, depth1 = (self._dense(a) for a in (gray0, depth0, gray1, depth1))
            self._follow_producer_stream(gray0, depth0, gray1, depth1)
            P, R, Cc = tuple(gray0.shape)
            dtype = self._batch_depth_type(depth0)
            if tuple(depth0.shape) != (P, R, Cc) or tuple(gray1.shape) != (P, R, Cc) or tuple(depth1.shape) != (P, R, Cc):
                raise ValueError("gray0, depth0, gray1 and depth1 must all be [P, rows, cols]")
            if self._batch_depth_type(depth1) != dtype:
                raise TypeError("depth1 must have the element type of depth0 (one depth type is passed for both)")
            self._check(self._L.phovo_batch_align_device_with_target_depth(
                self._h, P, R, Cc, gray0.data_ptr(), depth0.data_ptr(), dtype, float(depth_scale), gray1.data_ptr(),
                depth1.data_ptr(), None if initial_states is None else initial_states.data_ptr(),
                states_out.data_ptr(), iters_out.data_ptr()))
            return
        self._follow_producer_stream(gray0)
        P, R, Cc = tuple(gray0.shape)
        dtype = {torch.float64: capi.DEPTH_F64, torch.float32: capi.DEPTH_F32, torch.uint16: capi.DEPTH_U16,
                 torch.int16: capi.DEPTH_U16}[depth0.dtype]
        self._check(self._L.phovo_batch_align_device(self._h, P, R, Cc, gray0.data_ptr(), depth0.data_ptr(), dtype,
                                                     float(depth_scale), gray1.data_ptr(),
                                                     None if initial_states is None else initial_states.data_ptr(),
                                                     states_out.data_ptr(), iters_out.data_ptr()))

    def BatchWarpImage(self, gray0, depth0, rts, K, level=0, gray1=None, images=True, depth_scale=1.0):
        """WarpImage for P pairs in one call.  gray0 / gray1 u8 [P,R,C] and depth0 [P,R,C] (f64 / f32 metres or u16 raw *
        depth_scale), numpy or torch, all on the host or all on the device; rts [P,4,4] (numpy or torch).  Returns a dict:
        `warped` [P,R,C] u8 (None unless `images`), `diff` = |gray1 - warped| (None unless `images` and gray1 is given) --
        torch tensors on the device for device inputs, numpy otherwise -- and, as numpy [P], `num_landed` (source pixels
        that land in the target), `sum_abs_diff` (sum of |gray1 - warped| over them; None without gray1) and
        `mean_abs_diff` = sum_abs_diff / max(num_landed, 1)."""
        gray0, depth0, gray1 = (self._dense(a) for a in (gray0, depth0, gray1))
        P, R, Cc = tuple(gray0.shape)
        dtype = self._batch_depth_type(depth0)
        if tuple(depth0.shape) != (P, R, Cc) or (gray1 is not None and tuple(gray1.shape) != (P, R, Cc)):
            raise ValueError("gray0, depth0 and gray1 must all be [P, rows, cols]")
        on_device = not isinstance(gray0, np.ndarray) and gray0.is_cuda
        if on_device:
            self._follow_producer_stream(gray0)
        if getattr(rts, "is_cuda", False):
            import torch
            rts = rts.to(torch.float64).contiguous()
        else:
            rts = np.ascontiguousarray(np.asarray(rts), dtype=np.float64)
        if tuple(rts.shape) not in ((P, 4, 4), (P, 16)):
            raise ValueError("rts must be [P, 4, 4]")
        Kc = np.ascontiguousarray(K, dtype=np.float64).reshape(9)

        def image():
            if on_device:
                import torch
                return torch.empty((P, R, Cc), dtype=torch.uint8, device=gray0.device)
            return np.empty((P, R, Cc), np.uint8)
        warped = image() if images else None
        diff = image() if images and gray1 is not None else None
        landed = np.zeros(P, np.int32)
        sums = np.zeros(P, np.int64) if gray1 is not None else None
        self._check(self._L.phovo_batch_warp_image(self._h, P, R, Cc, capi._ptr(gray0), capi._ptr(depth0), dtype, float(depth_scale),
                                                   capi._ptr(rts), Kc.ctypes.data_as(capi._dp), int(level), capi._ptr(gray1),
                                                   capi._ptr(warped), capi._ptr(diff), landed.ctypes.data,
                                                   None if sums is None else sums.ctypes.data))
        return dict(warped=warped, diff=diff, num_landed=landed, sum_abs_diff=sums,
                    mean_abs_diff=None if sums is None else sums / np.maximum(landed, 1))

    def BatchEvalNormalEquations(self, gray0, depth0, gray1, states, level=0, depth_scale=1.0, depth1=None):
        """The normal equations of P pairs at the given states, at any pyramid level (built by the call, configured
        iterations or not): what EvalNormalEquations(level, states[p]) returns after SetSourceFrame(gray0[p], depth0[p])
        and SetTargetFrame(gray1[p]), to rounding.  gray0 / gray1 u8 [P,R,C] and depth0 [P,R,C] (f64 / f32 metres or
        u16 raw * depth_scale), numpy or torch, all on the host or all on the device; states [P,6] (numpy or torch).
        Returns a dict of numpy arrays: `H` [P,6,6] = J^T J (symmetric), `g` [P,6] = J^T r, `cost` [P] = 0.5 |r|^2 and
        `num_valid` [P].  J scales the image gradients by the configured imageGradientsScalingFactor and, in mode 0,
        carries the reference's temp11 term (AN:253): H is the solver's J^T J, not a calibrated information matrix.
        `depth1` [P,R,C] (target depth, depth0's element type) is what the photometric + depth solver (MODE_BIOBJECTIVE)
        needs: with it the results are EvalNormalEquations' after SetTargetFrame(gray1[p], depth1[p]) as well, i.e. of
        the stacked intensity + depth system; the other modes ignore it."""
        gray0, depth0, gray1, depth1 = (self._dense(a) for a in (gray0, depth0, gray1, depth1))
        P, R, Cc = tuple(gray0.shape)
        dtype = self._batch_depth_type(depth0)
        if tuple(depth0.shape) != (P, R, Cc) or tuple(gray1.shape) != (P, R, Cc):
            raise ValueError("gray0, depth0 and gray1 must all be [P, rows, cols]")
        if depth1 is not None:
            if tuple(depth1.shape) != (P, R, Cc):
                raise ValueError("depth1 must be [P, rows, cols] like depth0")
            if self._batch_depth_type(depth1) != dtype:
                raise TypeError("depth1 must have the element type of depth0 (one depth type is passed for both)")
        if not isinstance(gray0, np.ndarray) and gray0.is_cuda:
            self._follow_producer_stream(gray0)
        if getattr(states, "is_cuda", False):
            import torch
            states = states.to(torch.float64).contiguous()
        else:
            states = np.ascontiguousarray(np.asarray(states), dtype=np.float64)
        if tuple(states.shape) != (P, 6):
            raise ValueError("states must be [P, 6]")
        Hu = np.zeros((P, 21))
        g = np.zeros((P, 6))
        cost = np.zeros(P)
        nv = np.zeros(P, np.int32)
        if depth1 is not None:
            self._check(self._L.phovo_batch_eval_normal_equations_with_target_depth(
                self._h, P, R, Cc, capi._ptr(gray0), capi._ptr(depth0), dtype, float(depth_scale), capi._ptr(gray1),
                capi._ptr(depth1), capi._ptr(states), int(level), Hu.ctypes.data, g.ctypes.data, cost.ctypes.data, nv.ctypes.data))
        else:
            self._check(self._L.phovo_batch_eval_normal_equations(self._h, P, R, Cc, capi._ptr(gray0), capi._ptr(depth0), dtype,
                                                                  float(depth_scale), capi._ptr(gray1), capi._ptr(states), int(level),
                                                                  Hu.ctypes.data, g.ctypes.data, cost.ctypes.data, nv.ctypes.data))
        iu = np.triu_indices(6)
        H = np.zeros((P, 6, 6))
        H[:, iu[0], iu[1]] = Hu
        H[:, iu[1], iu[0]] = Hu
        return dict(H=H, g=g, cost=cost, num_valid=nv)

    @staticmethod
    def _dense(a):
        """A batch entry reads dense [P, rows, cols] frames: a strided numpy array or torch view is copied."""
        return None if a is None else np.ascontiguousarray(a) if isinstance(a, np.ndarray) else a.contiguous()

    @staticmethod
    def _batch_depth_type(depth0):
        if isinstance(depth0, np.ndarray):
            return {np.dtype(np.float64): capi.DEPTH_F64, np.dtype(np.float32): capi.DEPTH_F32,
                    np.dtype(np.uint16): capi.DEPTH_U16}[depth0.dtype]
        import torch
        return {torch.float64: capi.DEPTH_F64, torch.float32: capi.DEPTH_F32, torch.uint16: capi.DEPTH_U16,
                torch.int16: capi.DEPTH_U16}[depth0.dtype]

    def AlignSequence(self, gray, depth, depth_scale=1.0, diagnostics=False, information_level=None):
        """PhotoconsistencyVisualOdometry.cpp:212-259 for a whole recorded sequence in ONE batch call.

        The app aligns frame k-1 (source) to frame k (target) from a ZERO initial state every frame
        (VisualOdometry.cpp:175,224), so the N-1 alignments of a sequence are independent: the frames are
        uploaded once and pair k reads frames k and k+1 of the same device arrays.  `gray` [N,R,C] u8 and
        `depth` [N,R,C] (f64 / f32 metres or u16 raw * depth_scale), numpy or torch (host or device).
        Returns (states [N-1,6], iterations [N-1,MAXL], poses [N,4,4]) with poses[0] = I and
        poses[k] = poses[k-1] @ inv(Rt_k) as the app accumulates them (:234).
        With `diagnostics` a 4th element: BatchWarpImage's summary (num_landed, sum_abs_diff, mean_abs_diff [N-1]) of frame
        k-1 warped onto frame k with Rt_k at full resolution -- the |target - warped| image the app shows (:247-252),
        reduced to one number per frame.
        With `information_level` (a pyramid level) the 4th element is returned whether or not `diagnostics` is set and
        also carries BatchEvalNormalEquations' H [N-1,6,6], g, cost and num_valid of every pair at its solved state on
        that level: the solver's J^T J of each edge, for a pose graph or filter (scale it by a noise model)."""
        import torch
        dev = torch.device("cuda", torch.cuda.current_device())
        g = gray if isinstance(gray, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(gray))
        d = depth if isinstance(depth, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(depth))
        if d.dtype == torch.uint16:
            d = d.view(torch.int16)
        g, d = g.to(dev, non_blocking=True).contiguous(), d.to(dev, non_blocking=True).contiguous()
        n = g.shape[0]
        if n < 2:
            raise ValueError("a sequence needs at least two frames")
        states = torch.zeros((n - 1, 6), dtype=torch.float64, device=dev)
        iters = torch.zeros((n - 1, capi.MAXL), dtype=torch.int32, device=dev)
        self.SetStream(torch.cuda.current_stream(dev).cuda_stream)
        # the photometric + depth solver also reads the target depth: frame k+1's depth for pair k
        d1 = d[1:] if self.GetConfig().mode == capi.MODE_BIOBJECTIVE else None
        self.BatchAlignDevice(g[:-1], d[:-1], g[1:], states, iters, depth_scale=depth_scale, depth1=d1)   # overlapping views, no copies
        st, it = states.cpu().numpy(), iters.cpu().numpy()
        rts = np.stack([capi.state_to_rt(s) for s in st])
        poses = np.tile(np.eye(4), (n, 1, 1))
        for k in range(1, n):
            poses[k] = poses[k - 1] @ np.linalg.inv(rts[k - 1])
        if not diagnostics and information_level is None:
            return st, it, poses
        diag = {}
        if diagnostics:
            if getattr(self, "_K", None) is None:
                raise ValueError("diagnostics need SetIntrinsicMatrix")
            s = self.BatchWarpImage(g[:-1], d[:-1], rts, self._K, gray1=g[1:], images=False, depth_scale=depth_scale)
            diag.update({k: s[k] for k in ("num_landed", "sum_abs_diff", "mean_abs_diff")})
        if information_level is not None:
            diag.update(self.BatchEvalNormalEquations(g[:-1], d[:-1], g[1:], states, level=int(information_level),
                                                      depth_scale=depth_scale, depth1=d1))
        return st, it, poses, diag

    def BatchKernelTimes(self):
        """(pyramid_ms, align_ms) of the last BatchAlignDevice call, CUDA events on the context stream."""
        a, b = C.c_float(), C.c_float()
        self._check(self._L.phovo_batch_get_kernel_times(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def BatchSetRecordStats(self, enable):
        self._check(self._L.phovo_batch_set_record_stats(self._h, int(enable)))

    def BatchLastH2DBytes(self):
        """Bytes the last BatchAlign call with host inputs copied to the device."""
        n = C.c_uint64()
        self._check(self._L.phovo_batch_get_last_h2d_bytes(self._h, C.byref(n)))
        return int(n.value)

    def BatchSetDebugFlags(self, flags):
        """bit 0: exact warp for every pixel; bit 1: generic pixel bookkeeping (results must not change); bit 2 / bit 3: what the
        resident kernels do not take goes through the pool of per-pair contexts / the slot waves whatever the batch size."""
        self._check(self._L.phovo_batch_set_debug_flags(self._h, int(flags)))

    def BatchReleaseMemory(self):
        """Free what the batch entries keep between calls (level store, slot arena, pool contexts, pinned buffers)."""
        self._check(self._L.phovo_batch_release_memory(self._h))

    def BatchIterationStats(self, pair):
        out = []
        for i in range(self._L.phovo_batch_num_iter_stats(self._h, pair)):
            s = capi.IterStats()
            self._check(self._L.phovo_batch_get_iter_stats(self._h, pair, i, C.byref(s)))
            out.append(s.as_dict())
        return out

    # row-sharded single pair -------------------------------------------------------------------
    def ShardConfigure(self, rank, world):
        self._check(self._L.phovo_shard_configure(self._h, rank, world))

    def ShardBuffer(self):
        p = C.c_void_p()
        self._check(self._L.phovo_shard_buffer(self._h, C.byref(p)))
        return p.value

    def ShardReadBuffer(self):
        out = np.zeros(32)
        self._check(self._L.phovo_shard_read_buffer(self._h, out.ctypes.data_as(capi._dp)))
        return out

    def ShardWriteBuffer(self, values):
        v = np.ascontiguousarray(values, dtype=np.float64).reshape(32)
        self._check(self._L.phovo_shard_write_buffer(self._h, v.ctypes.data_as(capi._dp)))

    def ShardBegin(self):
        self._check(self._L.phovo_shard_begin(self._h))

    def ShardBeginLevel(self, level):
        self._check(self._L.phovo_shard_begin_level(self._h, level))

    def ShardPartial(self):
        self._check(self._L.phovo_shard_partial(self._h))

    def ShardStep(self, want_done=True):
        d = C.c_int32(0)
        self._check(self._L.phovo_shard_step(self._h, C.byref(d) if want_done else None))
        return bool(d.value)

    def ShardFinish(self):
        self._check(self._L.phovo_shard_finish(self._h))

    def ShardPeerExport(self):
        """64-byte CUDA IPC handle of this rank's exchange area (bytes)."""
        buf = C.create_string_buffer(64)
        self._check(self._L.phovo_shard_peer_export(self._h, buf))
        return buf.raw

    def ShardPeerImport(self, peer_rank, handle):
        self._check(self._L.phovo_shard_peer_import(self._h, int(peer_rank), C.c_char_p(bytes(handle))))

    def ShardPartialExchange(self):
        self._check(self._L.phovo_shard_partial_exchange(self._h))

    def ShardOptimize(self, min_shard_pixels=0):
        """The whole row-sharded Optimize() in one call: persistent kernel per level, sums exchanged inside the kernel
        over NVLink peer memory; levels below `min_shard_pixels` run unsharded on every rank."""
        self._check(self._L.phovo_shard_optimize(self._h, int(min_shard_pixels)))
