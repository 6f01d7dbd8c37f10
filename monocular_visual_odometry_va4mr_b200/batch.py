"""Batched per-frame hot path over independent sequences (BASELINE config 5).

``SequenceBatch`` wraps ``b200vo_batch_*`` (include/b200vo.h): per step and per sequence it
does what the reference's ``continuous_operation`` does on its hot path -- KLT on the landmark
keypoints and on the candidate keypoints (``VisualOdometryPipeLine.py:281,:287``), keep
``status == 1`` (``:282-284``), P3P-RANSAC + EPnP on the tracked landmarks (``:343``) -- for
``batch`` sequences in one set of kernel launches, with the previous frames' pyramids resident
in HBM.  torch is used only as a device-buffer allocator for the ``*_dev`` form.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import BatchCfg, c_f32p, c_f64p, c_i32p, c_u8p


def _p(a, t):
    return a.ctypes.data_as(t)


def _batch_K(K, batch):
    """K of a batch constructor: (3, 3) for every sequence, or (batch, 3, 3), one per sequence.  -> (the (3, 3) matrix that goes
    into the config, the (batch, 3, 3) rows to set afterwards or None)."""
    K = np.asarray(K, np.float64)
    if K.shape == (3, 3):
        return K, None
    if K.shape == (batch, 3, 3):
        return K[0], np.ascontiguousarray(K)
    raise ValueError(f"K must be (3, 3) or (batch = {batch}, 3, 3), got {K.shape}")


def _pinhole(K) -> bool:
    """What b200vo_*_set_intrinsics accepts (checked here where a refusal must come before another call)."""
    return bool(np.isfinite(K).all() and K[0, 0] > 0 and K[1, 1] > 0 and K[0, 1] == 0 and K[1, 0] == 0 and K[2, 0] == 0
                and K[2, 1] == 0 and K[2, 2] == 1)


def _set_intrinsics(ctx, fn, h, batch, seqs, K, what):
    """Shared body of SequenceBatch / VOBatch.set_intrinsics."""
    seqs = np.ascontiguousarray(seqs, np.int32).reshape(-1)
    K = np.ascontiguousarray(K, np.float64)
    if K.shape != (len(seqs), 3, 3):
        raise ValueError(f"K must be (len(seqs) = {len(seqs)}, 3, 3), got {K.shape}")
    rc = fn(h, len(seqs), _p(seqs, c_i32p), _p(K, c_f64p))
    if rc == -1:
        raise ValueError(f"{what}: {ctx.last_error()}")
    if rc != 0:
        raise _lib.B200VOError(f"{what} failed ({rc}): {ctx.last_error()}")


def _set_frame_size(ctx, fn, h, seqs, sizes, what):
    """Shared body of SequenceBatch / VOBatch.set_frame_size.  -> (seqs, sizes) as the call took them."""
    seqs = np.ascontiguousarray(seqs, np.int32).reshape(-1)
    sizes = np.asarray(sizes)
    if sizes.shape != (len(seqs), 2) or not np.issubdtype(sizes.dtype, np.integer):
        raise ValueError(f"sizes must be integer (len(seqs) = {len(seqs)}, 2) (rows, cols), got {sizes.dtype} {sizes.shape}")
    rows = np.ascontiguousarray(sizes[:, 0], np.int32)
    cols = np.ascontiguousarray(sizes[:, 1], np.int32)
    rc = fn(h, len(seqs), _p(seqs, c_i32p), _p(rows, c_i32p), _p(cols, c_i32p))
    if rc == -1:
        raise ValueError(f"{what}: {ctx.last_error()}")
    if rc != 0:
        raise _lib.B200VOError(f"{what} failed ({rc}): {ctx.last_error()}")
    return seqs, np.stack([rows, cols], 1)


def _pack_frames(frames, sizes, rows, cols, out=None):
    """A list of per-sequence 2-D uint8 images, each of its sequence's (rows_s, cols_s), packed into the slot layout
    (len, rows, cols); the bytes outside each image are zero.  An array is returned as it is."""
    if not isinstance(frames, (list, tuple)):
        return frames
    if len(frames) != len(sizes):
        raise ValueError(f"{len(frames)} frames for {len(sizes)} sequences")
    if out is None:
        out = np.zeros((len(frames), rows, cols), np.uint8)
    else:
        out[...] = 0
    for k, (f, (r, c)) in enumerate(zip(frames, sizes)):
        f = np.asarray(f)
        if f.dtype != np.uint8 or f.shape != (r, c):
            raise ValueError(f"frame {k} must be ({r}, {c}) uint8, got {f.dtype} {f.shape}")
        out[k, :r, :c] = f
    return out


class _PinnedBlock:
    """Owner of one b200vo_host_alloc block.  The numpy arrays carved from it keep it alive (it hangs off the
    ctypes buffer that is the arrays' base), so a result array that outlives its SequenceBatch -- e.g.
    ``SequenceBatch(...).step(...)['pose']`` -- never points into freed page-locked memory: the block is
    released when the LAST array referring to it is collected."""

    def __init__(self, ctx: _lib.Context, nbytes: int):
        self.ctx, self.nbytes = ctx, nbytes
        self.ptr = ctx.lib.b200vo_host_alloc(ctx.h, nbytes)
        if not self.ptr:
            raise MemoryError("b200vo_host_alloc")

    def array(self, shape, dtype) -> np.ndarray:
        dt = np.dtype(dtype)
        buf = (C.c_uint8 * self.nbytes).from_address(self.ptr)
        buf._owner = self          # ndarray.base -> memoryview -> buf -> this block
        return np.frombuffer(buf, dt, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            if self.ptr:
                # the context may already be closed: page-locked memory is freed all the same (ctx == NULL)
                self.ctx.lib.b200vo_host_free(self.ctx.h if getattr(self.ctx, "h", None) else None, self.ptr)
                self.ptr = None
        except Exception:
            pass


class SequenceBatch:
    def __init__(self, batch, rows, cols, K, win=(15, 15), max_level=5, criteria=(3, 50, 0.01),
                 min_eig_thr=1e-4, pnp_iters=500, pnp_reproj_err=8.0, pnp_conf=0.99,
                 max_landmarks=1024, max_candidates=1024, frame_size=None, ctx: _lib.Context | None = None):
        self.ctx = ctx or _lib.default_context(0)
        self.batch, self.rows, self.cols = int(batch), int(rows), int(cols)
        self.L, self.Cn = int(max_landmarks), int(max_candidates)
        self.frame_size = np.tile(np.int32([self.rows, self.cols]), (self.batch, 1))   # (batch, 2) rows, cols of every sequence
        self._submitted = []   # page-locked slot-layout copies of submitted frame lists, alive until their step
        cfg = BatchCfg()
        cfg.rows, cfg.cols = self.rows, self.cols
        cfg.win_w, cfg.win_h, cfg.max_level = int(win[0]), int(win[1]), int(max_level)
        cfg.crit_type, cfg.crit_max_count, cfg.crit_eps = int(criteria[0]), int(criteria[1]), float(criteria[2])
        cfg.min_eig_thr = float(min_eig_thr)
        cfg.pnp_iters, cfg.pnp_reproj_err, cfg.pnp_conf = int(pnp_iters), float(pnp_reproj_err), float(pnp_conf)
        K, K_rows = _batch_K(K, self.batch)
        Kf = K.reshape(9)
        for i in range(9):
            cfg.K[i] = float(Kf[i])
        cfg.max_landmarks, cfg.max_candidates = self.L, self.Cn
        self.cfg = cfg
        h = C.c_void_p()
        rc = self.ctx.lib.b200vo_batch_create(self.ctx.h, self.batch, C.byref(cfg), C.byref(h))
        if rc != 0:
            raise _lib.B200VOError(f"b200vo_batch_create failed ({rc}): {self.ctx.last_error()}")
        self.h = h
        if K_rows is not None:
            self.set_intrinsics(np.arange(self.batch), K_rows)
        if frame_size is not None:
            self.set_frame_size(np.arange(self.batch), frame_size)
        # host outputs (reused, page-locked so that step() reads them back without a staging copy)
        b, L, Cn = self.batch, self.L, self.Cn
        self.lm_next = self.pinned_empty((b, L, 2), np.float32)
        self.lm_status = self.pinned_empty((b, L), np.uint8)
        self.cand_next = self.pinned_empty((b, max(Cn, 1), 2), np.float32)
        self.cand_status = self.pinned_empty((b, max(Cn, 1)), np.uint8)
        self.pose = self.pinned_empty((b, 6), np.float64)
        self.pnp_ok = self.pinned_empty((b,), np.uint8)
        self.inlier_mask = self.pinned_empty((b, L), np.uint8)
        self.n_inliers = self.pinned_empty((b,), np.int32)
        # ctypes views of the reused result arrays, built once (step() is called thousands of times per second)
        self._out_ptrs = (_p(self.lm_next, c_f32p), _p(self.lm_status, c_u8p), _p(self.cand_next, c_f32p), _p(self.cand_status, c_u8p),
                          _p(self.pose, c_f64p), _p(self.pnp_ok, c_u8p), _p(self.inlier_mask, c_u8p), _p(self.n_inliers, c_i32p))
        self._out_dict = dict(lm_next=self.lm_next, lm_status=self.lm_status, cand_next=self.cand_next, cand_status=self.cand_status,
                              pose=self.pose, pnp_ok=self.pnp_ok, inlier_mask=self.inlier_mask, n_inliers=self.n_inliers)

    def close(self):
        """Destroys the device-side batch.  Page-locked arrays handed out by this object (step() results,
        pinned_empty / pinned_like / pinned_frames) stay valid for as long as they are referenced: each block is
        owned by its arrays (_PinnedBlock) and released with the last of them."""
        if getattr(self, "h", None):
            self.ctx.lib.b200vo_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc, what):
        if rc != 0:
            raise _lib.B200VOError(f"{what} failed ({rc}): {self.ctx.last_error()}")

    def set_intrinsics(self, seqs, K):
        """Give the distinct sequences ``seqs`` the camera matrices ``K`` (len(seqs), 3, 3); every later step poses them with
        their own K.  A K must be a pinhole camera: fx, fy finite and > 0, cx, cy finite, zero skew and other off-diagonal
        entries, last row (0, 0, 1).  Bad shapes, indices or matrices raise ValueError and change nothing.  Synchronous."""
        _set_intrinsics(self.ctx, self.ctx.lib.b200vo_batch_set_intrinsics, self.h, self.batch, seqs, K, "b200vo_batch_set_intrinsics")

    def set_frame_size(self, seqs, sizes):
        """Give the distinct sequences ``seqs`` the frame sizes ``sizes`` (len(seqs), 2) int (rows, cols).  ``rows`` x ``cols`` of the
        constructor is the slot, the largest frame: a sequence's image is the top-left of its slot in every frame array, and it is
        tracked and detected exactly as in a batch of its own size.  A size must fit the slot and exceed the window.  Bad shapes,
        indices or sizes, or submitted frames still waiting, raise ValueError and change nothing.  The next step needs prime().
        Synchronous."""
        seqs, sizes = _set_frame_size(self.ctx, self.ctx.lib.b200vo_batch_set_frame_size, self.h, seqs, sizes, "b200vo_batch_set_frame_size")
        self.frame_size[seqs] = sizes

    def _frames(self, frames):
        """frames of a step: the slot-layout array, or a list of per-sequence 2-D images packed into it"""
        return _pack_frames(frames, self.frame_size, self.rows, self.cols)

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array in page-locked host memory (b200vo_host_alloc): DMA'd in place by step()."""
        dt = np.dtype(dtype)
        nbytes = max(int(np.prod(shape)) * dt.itemsize, 1)
        return _PinnedBlock(self.ctx, nbytes).array(shape, dt)

    def pinned_like(self, arr: np.ndarray) -> np.ndarray:
        out = self.pinned_empty(arr.shape, arr.dtype)
        out[...] = arr
        return out

    def pinned_frames(self, n_sets: int = 1) -> np.ndarray:
        """(n_sets, batch, rows, cols) uint8 array in page-locked memory (b200vo_host_alloc)."""
        return self.pinned_empty((n_sets, self.batch, self.rows, self.cols), np.uint8)

    def prime(self, frames):
        frames = np.ascontiguousarray(self._frames(frames), np.uint8).reshape(self.batch, self.rows, self.cols)
        self._chk(self.ctx.lib.b200vo_batch_prime(self.h, _p(frames, c_u8p)), "b200vo_batch_prime")

    def submit_frames(self, frames):
        """Hand over the frames of a FUTURE step (page-locked array from pinned_frames(), or a list of per-sequence images,
        packed into a page-locked copy): their upload and pyramid build overlap the step in flight; the step called with
        frames=None consumes them."""
        if isinstance(frames, (list, tuple)):
            frames = _pack_frames(frames, self.frame_size, self.rows, self.cols, self.pinned_frames()[0])
            self._submitted = (self._submitted + [frames])[-3:]
        assert frames.dtype == np.uint8 and frames.flags.c_contiguous and frames.size == self.batch * self.rows * self.cols
        self._chk(self.ctx.lib.b200vo_batch_submit_frames(self.h, _p(frames, c_u8p)), "b200vo_batch_submit_frames")

    def submit_frames_dev(self, frames_dev: int):
        """The same look-ahead for frames already resident in device memory (int from tensor.data_ptr()): the
        pyramids are built beside the step in flight; step_dev(frames_dev=None, ...) consumes them."""
        self._chk(self.ctx.lib.b200vo_batch_submit_frames_dev(self.h, frames_dev), "b200vo_batch_submit_frames_dev")

    def step(self, frames, lm_pts, lm_obj, n_lm, cand_pts=None, n_cand=None):
        """Host buffers in, host buffers out (synchronous).  Returns a dict of views on REUSED page-locked arrays:
        the next step() overwrites them (copy what must survive it); they remain valid memory after close().
        frames=None: use the oldest frame set given to submit_frames()."""
        b, L, Cn = self.batch, self.L, self.Cn
        if frames is not None:
            frames = self._frames(frames)
        assert frames is None or (frames.dtype == np.uint8 and frames.flags.c_contiguous and frames.size == b * self.rows * self.cols)
        assert lm_pts.dtype == np.float32 and lm_pts.shape == (b, L, 2) and lm_pts.flags.c_contiguous
        assert lm_obj.dtype == np.float32 and lm_obj.shape == (b, L, 3) and lm_obj.flags.c_contiguous
        assert n_lm.dtype == np.int32 and n_lm.shape == (b,)
        if Cn > 0:
            assert cand_pts is not None and cand_pts.dtype == np.float32 and cand_pts.shape == (b, Cn, 2)
            assert n_cand is not None and n_cand.dtype == np.int32 and n_cand.shape == (b,)
        rc = self.ctx.lib.b200vo_batch_step(
            self.h, _p(frames, c_u8p) if frames is not None else None, _p(lm_pts, c_f32p), _p(lm_obj, c_f32p), _p(n_lm, c_i32p),
            _p(cand_pts, c_f32p) if Cn > 0 else None, _p(n_cand, c_i32p) if Cn > 0 else None, *self._out_ptrs)
        if rc != 0:
            # the counts are validated once, inside the call (a single sequence steps thousands of times per second)
            msg = self.ctx.last_error()
            if "is outside [0," in msg:
                raise ValueError(msg)
            self._chk(rc, "b200vo_batch_step")
        return self._out_dict

    def good_features(self, max_corners=1400, quality=0.1, min_dist=10.0):
        """cv2.goodFeaturesToTrack (reference :256) on the current frame of every sequence (the frames the last
        prime()/step() left resident).  -> (corners float32 (batch, max_corners, 2), n int32 (batch,)); row s holds
        n[s] corners in cv2's order."""
        corners = np.zeros((self.batch, int(max_corners), 2), np.float32)
        n = np.zeros(self.batch, np.int32)
        self._chk(self.ctx.lib.b200vo_batch_good_features(self.h, int(max_corners), float(quality), float(min_dist),
                                                          _p(corners, c_f32p), _p(n, c_i32p)), "b200vo_batch_good_features")
        return corners, n

    def step_dev(self, frames_dev, lm_pts_dev, lm_obj_dev, n_lm_dev, cand_pts_dev, n_cand_dev, out_dev: dict):
        """Device pointers in/out (ints from tensor.data_ptr()); asynchronous on the ctx stream.
        frames_dev=None: use the oldest frame set given to submit_frames_dev() / submit_frames()."""
        o = out_dev
        rc = self.ctx.lib.b200vo_batch_step_dev(
            self.h, frames_dev or None, lm_pts_dev, lm_obj_dev, n_lm_dev, cand_pts_dev, n_cand_dev,
            o["lm_next"], o["lm_status"], o["cand_next"], o["cand_status"], o["pose"], o["pnp_ok"],
            o["inlier_mask"], o["n_inliers"])
        self._chk(rc, "b200vo_batch_step_dev")


def _loop_cfg(rows, cols, K, options, max_landmarks, max_candidates, max_frames):
    o = options
    cfg = _lib.LoopCfg()
    bc = cfg.batch
    bc.rows, bc.cols = int(rows), int(cols)
    bc.win_w, bc.win_h, bc.max_level = int(o['winSize'][0]), int(o['winSize'][1]), int(o['maxLevel'])
    bc.crit_type, bc.crit_max_count, bc.crit_eps = int(o['criteria'][0]), int(o['criteria'][1]), float(o['criteria'][2])
    bc.min_eig_thr = 1e-4                          # cv2.calcOpticalFlowPyrLK's default (the reference passes none)
    bc.pnp_iters, bc.pnp_reproj_err, bc.pnp_conf = int(o['PnP_iterations']), float(o['PnP_error']), float(o['PnP_conf'])
    Kf = np.asarray(K, np.float64).reshape(9)   # the (3, 3) K of every sequence (per-sequence rows: VOBatch.set_intrinsics)
    for i in range(9):
        bc.K[i] = float(Kf[i])
    bc.max_landmarks, bc.max_candidates = int(max_landmarks), int(max_candidates)
    cfg.min_dist_landmarks, cfg.max_dist_landmarks = float(o['min_dist_landmarks']), float(o['max_dist_landmarks'])
    cfg.min_baseline_angle_deg, cfg.min_baseline_frames = float(o['min_baseline_angle']), int(o['min_baseline_frames'])
    if o.get('feature_block_size', 3) != 3 or o.get('feature_use_harris', False):
        raise NotImplementedError("VOBatch detects corners with blockSize 3 and no Harris detector (the reference's options)")
    cfg.max_corners, cfg.quality_level = int(o['feature_max_corners']), float(o['feature_quality_level'])
    cfg.feature_min_dist = float(o['feature_min_dist'])
    cfg.max_frames = int(max_frames)
    return cfg


class VOBatch:
    """The whole per-frame loop of the reference (``continuous_operation``, ``VisualOdometryPipeLine.py:326-373``) for
    ``batch`` independent sequences, with the VO state of every sequence resident on the device (``b200vo_loop_*``).

    ``options`` is the reference's option dict (main.py:20-44).  Each sequence is loaded once with the state its
    bootstrap produced (``initial_state``) and then advanced one frame per ``step``.  The state of a sequence is
    ``lm`` float32 (n_lm,3), ``lm_kp`` float32 (n_lm,2), the candidates ``keys`` / ``first_keys`` float32 (n_cand,2)
    and ``first_pose`` int32 (n_cand,), and ``poses`` float64 (n_poses,12) = ``self.transforms`` as (R_CW | t_CW).
    A sequence that cannot follow the reference's data flow stops with one of the status codes below and stays as it
    is until it is loaded again.  ``bootstrap`` runs the reference's bootstrap for any subset of the sequences on the
    device instead of ``load``; a sequence whose bootstrap finds no essential matrix gets ``NO_BOOTSTRAP``.

    ``K`` is the camera matrix of every sequence, (3, 3), or one per sequence, (batch, 3, 3).  ``set_intrinsics`` (or the
    ``K`` argument of ``load`` / ``bootstrap``) gives a slot another camera, e.g. when it is handed to a new sequence."""

    OK, IDLE, FEW_POINTS, PNP_FAILED, OVERFLOW, DETECT_LIMIT, NO_BOOTSTRAP = range(7)

    def __init__(self, batch, rows, cols, K, options, max_landmarks=4096, max_candidates=8192, max_frames=1024,
                 frame_size=None, ctx: _lib.Context | None = None):
        self.ctx = ctx or _lib.default_context(0)
        self.batch, self.rows, self.cols = int(batch), int(rows), int(cols)
        self.frame_size = np.tile(np.int32([self.rows, self.cols]), (self.batch, 1))   # (batch, 2) rows, cols of every sequence
        self._submitted = []
        self.L, self.Cn, self.P = int(max_landmarks), int(max_candidates), int(max_frames)
        self.options = options
        K, K_rows = _batch_K(K, self.batch)
        self.cfg = _loop_cfg(rows, cols, K, options, max_landmarks, max_candidates, max_frames)
        h = C.c_void_p()
        rc = self.ctx.lib.b200vo_loop_create(self.ctx.h, self.batch, C.byref(self.cfg), C.byref(h))
        if rc != 0:
            raise _lib.B200VOError(f"b200vo_loop_create failed ({rc}): {self.ctx.last_error()}")
        self.h = h
        if K_rows is not None:
            self.set_intrinsics(np.arange(self.batch), K_rows)
        if frame_size is not None:
            self.set_frame_size(np.arange(self.batch), frame_size)
        b = self.batch
        self._res = dict(status=self.pinned_empty((b,), np.int32), n_inliers=self.pinned_empty((b,), np.int32),
                         n_lm=self.pinned_empty((b,), np.int32), n_cand=self.pinned_empty((b,), np.int32),
                         pose_cw=self.pinned_empty((b, 12), np.float64))
        r = self._res
        self._res_ptrs = (_p(r['status'], c_i32p), _p(r['n_inliers'], c_i32p), _p(r['n_lm'], c_i32p), _p(r['n_cand'], c_i32p),
                          _p(r['pose_cw'], c_f64p))

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.b200vo_loop_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc, what):
        if rc == -1:
            raise ValueError(f"{what}: {self.ctx.last_error()}")
        if rc != 0:
            raise _lib.B200VOError(f"{what} failed ({rc}): {self.ctx.last_error()}")

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array in page-locked host memory (b200vo_host_alloc)."""
        dt = np.dtype(dtype)
        return _PinnedBlock(self.ctx, max(int(np.prod(shape)) * dt.itemsize, 1)).array(shape, dt)

    def pinned_frames(self, n_sets: int = 1) -> np.ndarray:
        """(n_sets, batch, rows, cols) uint8 array in page-locked memory, for submit_frames() and step()."""
        return self.pinned_empty((n_sets, self.batch, self.rows, self.cols), np.uint8)

    def set_intrinsics(self, seqs, K):
        """Give the distinct sequences ``seqs`` the camera matrices ``K`` (len(seqs), 3, 3): every later step and bootstrap of
        those sequences tracks, poses and triangulates with their own K.  A K must be a pinhole camera: fx, fy finite and > 0,
        cx, cy finite, zero skew and other off-diagonal entries, last row (0, 0, 1).  The sequences' states, status and frames
        are not touched: to hand a slot to a sequence of another camera, set its K just before ``load`` or ``bootstrap`` (or
        pass ``K`` to them).  Bad shapes, indices or matrices raise ValueError and change nothing.  Synchronous."""
        _set_intrinsics(self.ctx, self.ctx.lib.b200vo_loop_set_intrinsics, self.h, self.batch, seqs, K, "b200vo_loop_set_intrinsics")

    def set_frame_size(self, seqs, sizes):
        """Give the distinct sequences ``seqs`` the frame sizes ``sizes`` (len(seqs), 2) int (rows, cols).  ``rows`` x ``cols`` of the
        constructor is the slot, the largest frame: a sequence's image is the top-left of its slot in the frames of ``step``,
        ``submit_frames`` and ``bootstrap`` (which also take a list of per-sequence images), and each sequence runs exactly as in
        a batch of its own size.  The listed sequences become IDLE (state kept, skipped by ``step``) until ``load`` or
        ``bootstrap``.  A size must fit the slot and exceed the window.  Bad shapes, indices or sizes, or submitted frames
        still waiting, raise ValueError and change nothing.  Synchronous."""
        seqs, sizes = _set_frame_size(self.ctx, self.ctx.lib.b200vo_loop_set_frame_size, self.h, seqs, sizes, "b200vo_loop_set_frame_size")
        self.frame_size[seqs] = sizes

    def load(self, seq: int, frame: np.ndarray, state: dict, K=None):
        """Set sequence ``seq`` to ``state`` (see the class docstring) with ``frame`` as its current frame; its status
        becomes OK.  ``K`` (3, 3): the sequence's camera from now on (``set_intrinsics`` first).  Out-of-range counts or
        first_pose values raise ValueError and change nothing."""
        f = np.ascontiguousarray(frame, np.uint8)
        if not 0 <= int(seq) < self.batch:
            raise ValueError(f"seq = {seq} is outside [0, batch = {self.batch})")
        r, c = (int(v) for v in self.frame_size[int(seq)])
        if f.shape != (r, c):
            raise ValueError(f"frame must be ({r}, {c}) uint8: the sequence's frame size")
        lm = np.ascontiguousarray(state['lm'], np.float32).reshape(-1, 3)
        kp = np.ascontiguousarray(state['lm_kp'], np.float32).reshape(-1, 2)
        keys = np.ascontiguousarray(state['keys'], np.float32).reshape(-1, 2)
        fk = np.ascontiguousarray(state['first_keys'], np.float32).reshape(-1, 2)
        fp = np.ascontiguousarray(state['first_pose'], np.int32).reshape(-1)
        poses = np.ascontiguousarray(state['poses'], np.float64).reshape(-1, 12)
        if len(kp) != len(lm) or len(fk) != len(keys) or len(fp) != len(keys):
            raise ValueError("lm / lm_kp and keys / first_keys / first_pose must have one row per point")
        if K is not None:
            K = np.asarray(K, np.float64)
            if K.shape != (3, 3) or not _pinhole(K):
                raise ValueError("K must be a (3, 3) pinhole camera matrix (see set_intrinsics)")
        self._chk(self.ctx.lib.b200vo_loop_load(self.h, int(seq), _p(f, c_u8p), _p(lm, c_f32p), _p(kp, c_f32p), len(lm),
                                                _p(keys, c_f32p), _p(fk, c_f32p), _p(fp, c_i32p), len(keys), _p(poses, c_f64p),
                                                len(poses)), "b200vo_loop_load")
        if K is not None:   # after the load, which is the call that can still refuse
            self.set_intrinsics([seq], K[None])

    def bootstrap(self, frames0, frames1, seqs=None, K=None) -> dict:
        """The reference's bootstrap (``initialization``) on the device for the sequences ``seqs`` (distinct indices; None:
        every sequence) from their two bootstrap frames ``frames0`` / ``frames1`` (len(seqs), rows, cols) uint8, with the
        ratio ``options['feature_ratio']``.  A sequence that succeeds ends up exactly as ``load(s, frames1[k],
        initial_state(K, options, *match_bootstrap_frames(frames0[k], frames1[k], ratio)))`` leaves it.  Returns int32
        arrays (len(seqs),): ``status`` (OK, NO_BOOTSTRAP or OVERFLOW), ``num_pts`` (the essential-matrix inlier count),
        ``n_lm`` and ``n_cand``.  A failing sequence keeps its state and is skipped by ``step`` until it is loaded or
        bootstrapped again.  ``K`` (len(seqs), 3, 3): the listed sequences' cameras from now on (``set_intrinsics`` first).
        Bad indices, frame shapes or K raise ValueError and change nothing.  Synchronous."""
        seqs = np.arange(self.batch, dtype=np.int32) if seqs is None else np.ascontiguousarray(seqs, np.int32).reshape(-1)
        if isinstance(frames0, (list, tuple)) or isinstance(frames1, (list, tuple)):
            if ((seqs < 0) | (seqs >= self.batch)).any():
                raise ValueError(f"seqs must lie in [0, batch = {self.batch})")
            frames0 = _pack_frames(list(frames0), self.frame_size[seqs], self.rows, self.cols)
            frames1 = _pack_frames(list(frames1), self.frame_size[seqs], self.rows, self.cols)
        f0 = np.ascontiguousarray(frames0, np.uint8)
        f1 = np.ascontiguousarray(frames1, np.uint8)
        shape = (len(seqs), self.rows, self.cols)
        if f0.shape != shape or f1.shape != shape:
            raise ValueError(f"frames0 and frames1 must be {shape} uint8")
        if K is not None:
            self.set_intrinsics(seqs, K)
        n = len(seqs)
        out = {k: np.zeros(max(n, 1), np.int32) for k in ('status', 'num_pts', 'n_lm', 'n_cand')}
        self._chk(self.ctx.lib.b200vo_loop_bootstrap(self.h, n, _p(seqs, c_i32p), _p(f0, c_u8p), _p(f1, c_u8p),
                                                     float(self.options['feature_ratio']), *(_p(out[k], c_i32p) for k in out)),
                  "b200vo_loop_bootstrap")
        return {k: v[:n] for k, v in out.items()}

    def read_state(self, seq: int) -> dict:
        """The state of sequence ``seq`` (copies) and its ``status``."""
        lm = np.zeros((self.L, 3), np.float32)
        kp = np.zeros((self.L, 2), np.float32)
        keys = np.zeros((self.Cn, 2), np.float32)
        fk = np.zeros((self.Cn, 2), np.float32)
        fp = np.zeros(self.Cn, np.int32)
        poses = np.zeros((self.P, 12), np.float64)
        n_lm, n_cand, n_poses, status = (C.c_int32(0) for _ in range(4))
        self._chk(self.ctx.lib.b200vo_loop_read_state(self.h, int(seq), _p(lm, c_f32p), _p(kp, c_f32p), C.byref(n_lm), _p(keys, c_f32p),
                                                      _p(fk, c_f32p), _p(fp, c_i32p), C.byref(n_cand), _p(poses, c_f64p),
                                                      C.byref(n_poses), C.byref(status)), "b200vo_loop_read_state")
        nl, nc, npo = n_lm.value, n_cand.value, n_poses.value
        return dict(lm=lm[:nl], lm_kp=kp[:nl], keys=keys[:nc], first_keys=fk[:nc], first_pose=fp[:nc], poses=poses[:npo],
                    status=status.value)

    def _list(self, seqs) -> np.ndarray:
        """The sequences of a listed step as int32 (n,); ValueError unless they are 1 to batch distinct indices in [0, batch)."""
        a = np.asarray(seqs)
        if a.ndim != 1 or a.size < 1 or a.size > self.batch or not np.issubdtype(a.dtype, np.integer):
            raise ValueError(f"seqs must be 1 to batch = {self.batch} integer sequence indices, got {a.dtype} {a.shape}")
        if ((a < 0) | (a >= self.batch)).any():
            raise ValueError(f"seqs must lie in [0, batch = {self.batch})")
        if len(np.unique(a)) != len(a):
            raise ValueError("seqs must be distinct")
        return np.ascontiguousarray(a, np.int32)

    def _listed_frames(self, frames, seqs, out=None) -> np.ndarray:
        """frames of a listed step: (len(seqs), rows, cols) uint8 in the slot layout, or a list of the listed sequences' images"""
        frames = _pack_frames(frames, self.frame_size[seqs], self.rows, self.cols, out)
        if not isinstance(frames, np.ndarray) or frames.dtype != np.uint8 or frames.shape != (len(seqs), self.rows, self.cols):
            raise ValueError(f"frames must be ({len(seqs)}, {self.rows}, {self.cols}) uint8 or a list of {len(seqs)} images")
        return np.ascontiguousarray(frames)

    def submit_frames(self, frames, seqs=None):
        """Frames of a FUTURE step (page-locked, from pinned_frames(), or a list of per-sequence images, packed into a page-locked
        copy); step(None) consumes them, oldest first.  ``seqs``: the frames of a listed step (see ``step``), consumed by
        ``step(None, seqs)`` with the same list."""
        if seqs is not None:
            seqs = self._list(seqs)
            if isinstance(frames, (list, tuple)):
                frames = self._listed_frames(frames, seqs, self.pinned_empty((len(seqs), self.rows, self.cols), np.uint8))
                self._submitted = (self._submitted + [frames])[-3:]
            else:
                frames = self._listed_frames(frames, seqs)
            self._chk(self.ctx.lib.b200vo_loop_submit_frames_seqs(self.h, len(seqs), _p(seqs, c_i32p), _p(frames, c_u8p)),
                      "b200vo_loop_submit_frames_seqs")
            return
        if isinstance(frames, (list, tuple)):
            frames = _pack_frames(frames, self.frame_size, self.rows, self.cols, self.pinned_frames()[0])
            self._submitted = (self._submitted + [frames])[-3:]
        assert frames.dtype == np.uint8 and frames.flags.c_contiguous and frames.size == self.batch * self.rows * self.cols
        self._chk(self.ctx.lib.b200vo_loop_submit_frames(self.h, _p(frames, c_u8p)), "b200vo_loop_submit_frames")

    def submit_frames_dev(self, frames_dev: int, seqs=None):
        """The same for frames resident in device memory (int from tensor.data_ptr()); step_dev(None, ...) consumes them.
        ``seqs``: (len(seqs), rows, cols) frames of a listed step, consumed by ``step_dev(None, out_dev, seqs)``."""
        if seqs is not None:
            seqs = self._list(seqs)
            self._chk(self.ctx.lib.b200vo_loop_submit_frames_seqs_dev(self.h, len(seqs), _p(seqs, c_i32p), frames_dev),
                      "b200vo_loop_submit_frames_seqs_dev")
            return
        self._chk(self.ctx.lib.b200vo_loop_submit_frames_dev(self.h, frames_dev), "b200vo_loop_submit_frames_dev")

    def step(self, frames=None, seqs=None) -> dict:
        """One frame for every sequence (frames (batch, rows, cols) uint8 in the slot layout, or a list of per-sequence images;
        None: the oldest submitted set).  Synchronous.
        Returns views on REUSED page-locked arrays: status, n_inliers, n_lm, n_cand int32 (batch,) and pose_cw float64
        (batch, 12), the pose appended this step (0 unless status is OK).

        ``seqs``: a listed step that advances only the distinct sequences ``seqs`` (any order), e.g. the streams that have a
        new frame this tick.  frames are then (len(seqs), rows, cols) or a list of the listed sequences' images, in list
        order; None consumes a set submitted with the same list.  Each listed sequence runs exactly the step it runs in a
        batch of its own; the others are not touched and resume from their current frame when they are listed again.  The
        results are the first len(seqs) rows of the same arrays, in list order.  Bad shapes or indices raise ValueError."""
        if seqs is not None:
            seqs = self._list(seqs)
            n = len(seqs)
            if frames is not None:
                frames = self._listed_frames(frames, seqs)
            self._chk(self.ctx.lib.b200vo_loop_step_seqs(self.h, n, _p(seqs, c_i32p), _p(frames, c_u8p) if frames is not None else None,
                                                         *self._res_ptrs), "b200vo_loop_step_seqs")
            return {k: v[:n] for k, v in self._res.items()}
        if frames is not None:
            frames = np.ascontiguousarray(_pack_frames(frames, self.frame_size, self.rows, self.cols), np.uint8)
            assert frames.size == self.batch * self.rows * self.cols
        self._chk(self.ctx.lib.b200vo_loop_step(self.h, _p(frames, c_u8p) if frames is not None else None, *self._res_ptrs),
                  "b200vo_loop_step")
        return self._res

    def step_dev(self, frames_dev, out_dev: dict, seqs=None):
        """Device pointers (ints from tensor.data_ptr()) for the frames (None: the oldest submitted set) and for the results
        ``status``, ``n_inliers``, ``n_lm``, ``n_cand`` (int32 (batch,)) and ``pose_cw`` (float64 (batch, 12)).
        Asynchronous on the ctx stream.  ``seqs``: a listed step (see ``step``): frames_dev holds (len(seqs), rows, cols),
        and the results fill the first len(seqs) rows in list order."""
        o = out_dev
        if seqs is not None:
            seqs = self._list(seqs)
            self._chk(self.ctx.lib.b200vo_loop_step_seqs_dev(self.h, len(seqs), _p(seqs, c_i32p), frames_dev or None, o['status'],
                                                             o['n_inliers'], o['n_lm'], o['n_cand'], o['pose_cw']),
                      "b200vo_loop_step_seqs_dev")
            return
        self._chk(self.ctx.lib.b200vo_loop_step_dev(self.h, frames_dev or None, o['status'], o['n_inliers'], o['n_lm'], o['n_cand'],
                                                    o['pose_cw']), "b200vo_loop_step_dev")


def match_bootstrap_frames(frame0, frame1, ratio=0.8):
    """The reference's bootstrap matching (``VisualOdometryPipeLine.py:209-245``) on the CUDA path: SIFT
    detectAndCompute on both frames, knnMatch(k=2) and the ratio test.  -> (pts0, pts1) float32 (n, 2)."""
    from . import cv2_compat
    sift = cv2_compat.SIFT_create()
    kp0, d0 = sift.detectAndCompute(frame0, None)
    kp1, d1 = sift.detectAndCompute(frame1, None)
    good = [m for m, n in cv2_compat.BFMatcher().knnMatch(d0, d1, k=2) if m.distance < ratio * n.distance]
    pts0 = np.float32([kp0[m.queryIdx].pt for m in good]).reshape(-1, 2)
    pts1 = np.float32([kp1[m.trainIdx].pt for m in good]).reshape(-1, 2)
    return pts0, pts1


def initial_state(K, options, first_keys, keys) -> dict:
    """The state ``initialization`` (:295-330) leaves behind, from the bootstrap matches: findEssentialMat -> inlier split
    -> recoverPose -> t * sign(t_z) (:317) -> triangulation of the inliers against the first pose (I, 0).
    -> a state dict for ``VOBatch.load`` (two poses), plus ``num_pts`` = the essential-matrix inlier count."""
    from . import cv2_compat, hotpath
    K = np.asarray(K, np.float64).reshape(3, 3)
    first_keys = np.ascontiguousarray(first_keys, np.float32).reshape(-1, 2)
    keys = np.ascontiguousarray(keys, np.float32).reshape(-1, 2)
    E, mask = cv2_compat.findEssentialMat(first_keys, keys, K, method=cv2_compat.RANSAC, prob=0.99, threshold=1.0)
    if E is None:
        raise ValueError("findEssentialMat found no essential matrix in the bootstrap matches")
    inl = mask.ravel() == 1
    pf, pk = first_keys[inl], keys[inl]
    pt = np.zeros(len(pk), np.int32)
    _, R, t, _ = cv2_compat.recoverPose(E, pf, pk, K)
    t = t * np.sign(t[2])
    poses = hotpath.pack_poses([(np.eye(3), np.zeros((3, 1))), (R, t)])
    too_short, lm, lm_kp = hotpath.triangulate_landmarks(K, options, pf, pk, pt, poses[:1], R, t)
    return dict(lm=lm, lm_kp=lm_kp, keys=pk[too_short], first_keys=pf[too_short], first_pose=pt[too_short], poses=poses,
                num_pts=int(inl.sum()))
