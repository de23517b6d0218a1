"""Batched, GPU-resident VO driver (SURVEY §8f row N2): the reference's per-frame loop — track against the current
keyframe, keyframe policy, pose chaining, TUM pose file, keyframe-id file (pose_est_tools.py:1416-1628) — on top of the
front-end's keyframe mode.

The reference handles one frame per Python iteration.  Here a whole batch of frames is tracked SPECULATIVELY against
the current keyframe in one captured kernel chain; the host then walks the batch in frame order with the reference's
keyframe policy.  When frame j becomes a keyframe, its store slot is promoted on the device and only stage B (temporal
matching, RANSAC, refinement) is re-run for the frames after j — their remap / stereo matching / triangulation is
reused.  The sequence of poses and keyframes is the one the sequential loop produces.

The same driver runs the RGB-D front-end (an RgbdFrontendConfig): one camera, depth maps and keypoints per frame.
"""
from __future__ import annotations

import math
import os
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field
from typing import Iterable, List, Optional, Sequence

import numpy as np
import torch

from . import ops
from .frontend import Frontend, FrontendConfig, RgbdFrontendConfig

INPUT_KEYS = ("omni", "px_top", "desc_top", "boff_top", "px_bot", "desc_bot", "boff_bot")
RGBD_INPUT_KEYS = ("depth", "px", "desc", "n_kp")


# ---------------------------------------------------------------------------------------------------------------------
# host-side pieces of run_VO
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class KeyframePolicy:
    """Thresholds of run_VO (pose_est_tools.py:1296-1309); the defaults are its indoor set."""
    pos_min: float = 0.01                       # [m]
    pos_max: float = 0.20
    ang_min: float = math.radians(1.0)
    ang_max: float = math.radians(10.0)
    tracked_ratio: float = 0.10                 # vs the running average of tracked correspondences
    keypoint_ratio: float = 0.10                # vs the keyframe's number of valid keypoints

    @classmethod
    def outdoors(cls) -> "KeyframePolicy":
        return cls(pos_min=0.1, pos_max=0.20, ang_min=math.radians(1.0), ang_max=math.radians(4.0))

    def wants_keyframe(self, dist: float, angle: float, num_tracked: float, prev_avg: float, n_kp_frame: int,
                       n_kp_keyframe: int) -> bool:
        """The decision tree of pose_est_tools.py:1519-1537, including its rotation branch, which compares the
        translation ceiling with the rotation ceiling (`pos_max < ang_max`) and therefore never fires with the
        reference's own thresholds — reproduced as is."""
        by_pos = self.pos_min < dist < self.pos_max
        by_ang = self.ang_min < angle < self.ang_max
        if not (by_pos or by_ang):
            return False
        if not (num_tracked > self.tracked_ratio * prev_avg and n_kp_frame > self.keypoint_ratio * n_kp_keyframe):
            return False
        if by_pos:
            return angle < self.ang_max
        if self.ang_min < angle:
            return dist < self.pos_max < self.ang_max
        return False


def translation_metric(T: np.ndarray) -> float:
    """transformations.rpe_translation_metric (transformations.py:2078-2084)."""
    return float(np.linalg.norm(T[:3, 3]))


def rotation_metric(T: np.ndarray) -> float:
    """transformations.rpe_rotation_metric (transformations.py:2097-2106)."""
    return float(np.arccos(min(1.0, max(-1.0, 0.5 * (np.trace(T[:3, :3]) - 1.0)))))


def quaternion_wxyz(T: np.ndarray) -> np.ndarray:
    """Unit quaternion [w, x, y, z] of the rotation block, w >= 0: the dominant eigenvector of the symmetric 4x4 matrix
    built from R, as transformations.quaternion_from_matrix(isprecise=False) computes it (transformations.py:1311-1332)."""
    R = np.asarray(T, np.float64)[:3, :3]
    K = np.zeros((4, 4))
    K[0, 0] = R[0, 0] - R[1, 1] - R[2, 2]
    K[1, 1] = R[1, 1] - R[0, 0] - R[2, 2]
    K[2, 2] = R[2, 2] - R[0, 0] - R[1, 1]
    K[3, 3] = R[0, 0] + R[1, 1] + R[2, 2]
    K[1, 0] = R[0, 1] + R[1, 0]
    K[2, 0] = R[0, 2] + R[2, 0]
    K[2, 1] = R[1, 2] + R[2, 1]
    K[3, 0] = R[2, 1] - R[1, 2]
    K[3, 1] = R[0, 2] - R[2, 0]
    K[3, 2] = R[1, 0] - R[0, 1]
    w, V = np.linalg.eigh(K / 3.0)  # eigh reads the lower triangle
    q = V[[3, 0, 1, 2], int(np.argmax(w))]
    return -q if q[0] < 0.0 else q


def tum_line(frame_id, T: np.ndarray) -> str:
    """One line of the estimated-poses file: `id tx ty tz qx qy qz qw` (pose_est_tools.py:1609-1612)."""
    q = quaternion_wxyz(T)
    t = np.asarray(T, np.float64)[:3, 3]
    return " ".join(str(v) for v in (frame_id, t[0], t[1], t[2], q[1], q[2], q[3], q[0]))


@dataclass
class VOResult:
    frame_ids: List[int] = field(default_factory=list)
    poses_wrt_S: List[np.ndarray] = field(default_factory=list)          # T_C_curr_frame_wrt_S_est per frame, 4x4 [m]
    poses_wrt_keyframe: List[np.ndarray] = field(default_factory=list)   # T_frame_wrt_tracking_ref_frame, 4x4 [m]
    parent_ids: List[int] = field(default_factory=list)
    keyframe_ids: List[int] = field(default_factory=list)
    tracked: List[int] = field(default_factory=list)                     # RANSAC inliers per frame (0 for keyframe 0)
    status: str = "ok"
    device_steps: int = 0
    device_retracks: int = 0


class TrackingState:
    """The bookkeeping of run_VO between frames (pose_est_tools.py:1403-1411, 1489-1566), one call per frame."""

    def __init__(self, policy: KeyframePolicy, number_of_cams: int = 2, units_to_m: float = 1.0):
        self.policy, self.number_of_cams, self.units_to_m = policy, number_of_cams, units_to_m
        self.T_key_wrt_S: List[np.ndarray] = []
        self.T_curr_wrt_S = np.eye(4)
        self.keyframe_id: Optional[int] = None
        self.keyframe_kp = 0
        self.tracked_since_keyframe = 0
        self.prev_avg = 0.0
        self.result = VOResult()

    def _record(self, frame_id, T_rel, inliers):
        r = self.result
        r.frame_ids.append(frame_id)
        r.poses_wrt_S.append(self.T_curr_wrt_S.copy())
        r.poses_wrt_keyframe.append(T_rel.copy())
        r.parent_ids.append(self.keyframe_id if self.keyframe_id is not None else frame_id)
        r.tracked.append(int(inliers))

    def _make_keyframe(self, frame_id, T_rel, n_kp):
        # pose_est_tools.py:1553-1566
        if self.T_key_wrt_S:
            self.T_key_wrt_S.append(self.T_key_wrt_S[-1] @ T_rel)
        else:
            self.T_key_wrt_S.append(self.T_curr_wrt_S.copy())
        self.keyframe_id, self.keyframe_kp = frame_id, n_kp
        self.tracked_since_keyframe, self.prev_avg = 0, 0.0
        self.result.keyframe_ids.append(frame_id)

    def first_frame(self, frame_id, n_kp):
        self._record(frame_id, np.eye(4), 0)
        self._make_keyframe(frame_id, np.eye(4), n_kp)

    def tracked_frame(self, frame_id, pose34: np.ndarray, inliers: int, n_kp: int) -> bool:
        """Feed the front-end's result for `frame_id` (pose of the frame wrt the keyframe in model units, RANSAC
        inliers, valid keypoints).  Returns True when the frame became the new keyframe."""
        T_rel = np.eye(4)
        T_rel[:3] = np.asarray(pose34, np.float64).reshape(3, 4)
        T_rel[:3, 3] *= self.units_to_m                       # pose_est_tools.py:833
        self.T_curr_wrt_S = self.T_key_wrt_S[-1] @ T_rel       # pose_est_tools.py:837
        self.tracked_since_keyframe += 1
        num_tracked = inliers / float(self.number_of_cams)    # pose_est_tools.py:1513
        create = self.policy.wants_keyframe(translation_metric(T_rel), rotation_metric(T_rel), num_tracked, self.prev_avg,
                                            n_kp, self.keyframe_kp)
        self.prev_avg = (num_tracked + (self.tracked_since_keyframe - 1.0) * self.prev_avg) / self.tracked_since_keyframe
        self._record(frame_id, T_rel, inliers)
        if create:
            self._make_keyframe(frame_id, T_rel, n_kp)
        return create


# ---------------------------------------------------------------------------------------------------------------------
# the batched driver
# ---------------------------------------------------------------------------------------------------------------------
def frontend_layout(cfg):
    """What the driver takes from the kind of front-end: (input keys, {key: (batch shape, dtype)}, number_of_cams,
    default minimum of correspondences).  The trackers refuse fewer than 2 * 3 * 0.33 * 2 (TrackerStereoSE3,
    pose_est_tools.py:779-781) or 2 * 3 * 1 (TrackerRGBDSE3.track_frame) correspondences."""
    c = cfg
    if isinstance(cfg, RgbdFrontendConfig):
        return RGBD_INPUT_KEYS, {
            "depth": ((c.batch, c.height, c.width), torch.float32),
            "px": ((c.batch, c.max_kp, 2), torch.float32),
            "desc": ((c.batch, c.max_kp, 32), torch.uint8),
            "n_kp": ((c.batch,), torch.int32),
        }, 1, 2 * 3 * 1
    return INPUT_KEYS, {
        "omni": ((c.batch, c.src_h, c.src_w, c.channels), torch.uint8),
        "px_top": ((c.batch, c.max_feat_per_view, 2), torch.float32),
        "px_bot": ((c.batch, c.max_feat_per_view, 2), torch.float32),
        "desc_top": ((c.batch, c.max_feat_per_view, 32), torch.uint8),
        "desc_bot": ((c.batch, c.max_feat_per_view, 32), torch.uint8),
        "boff_top": ((c.batch, c.n_buckets + 1), torch.int32),
        "boff_bot": ((c.batch, c.n_buckets + 1), torch.int32),
    }, 2, 2 * 3 * (0.33 * 2)


class BatchedVO:
    """frames: sequence of per-frame dicts with the front-end's inputs for ONE frame each: SOS (FrontendConfig)
    omni [H,W,C] u8, px_* [F,2] f32, desc_* [F,32] u8, boff_* [n_buckets+1] i32; RGB-D (RgbdFrontendConfig, lut None)
    depth [height,width] f32, px [max_kp,2] f32, desc [max_kp,32] u8, n_kp (int)."""

    def __init__(self, ctx: ops.Context, cfg, lut: Optional[torch.Tensor], hyp: torch.Tensor,
                 policy: Optional[KeyframePolicy] = None, units_to_m: float = 1.0, min_correspondences: Optional[int] = None):
        if not cfg.keyframe_mode:
            raise ValueError("BatchedVO needs a front-end configuration with keyframe_mode=True")
        self.ctx, self.cfg = ctx, cfg
        self.fe = Frontend(ctx, cfg, lut, hyp)
        self.policy = policy or KeyframePolicy()
        self.units_to_m = units_to_m
        self.input_keys, shapes, self.number_of_cams, default_min = frontend_layout(cfg)
        self._step = self.fe.step_rgbd if isinstance(cfg, RgbdFrontendConfig) else self.fe.step
        self.min_correspondences = default_min if min_correspondences is None else min_correspondences
        # pinned staging (one batch) + its device twin; frames are packed into the staging arrays on the host
        # two sets, so that the next batch is packed while the current one is copied, tracked and resolved
        self._pinned = [{k: torch.zeros(shape, dtype=dt).pin_memory() for k, (shape, dt) in shapes.items()} for _ in range(2)]
        self._host = [{k: v.numpy() for k, v in p.items()} for p in self._pinned]
        self._dev = [{k: v.to(ctx.device) for k, v in p.items()} for p in self._pinned]
        self._pool = ThreadPoolExecutor(max_workers=max(1, min(16, len(os.sched_getaffinity(0)))))
        self._prefetch = ThreadPoolExecutor(max_workers=1)

    def close(self):
        self._prefetch.shutdown(wait=True)
        self._pool.shutdown(wait=True)
        self.fe.close()

    def _pack(self, frames: Sequence[dict], s: int):
        """Frames into the pinned staging set s (host only)."""
        B = self.cfg.batch
        assert len(frames) <= B
        host = self._host[s]

        def pack(i):                        # numpy copies release the GIL
            for k in self.input_keys:
                host[k][i] = frames[i][k]
        # packing a batch of images is the driver's largest host cost (118 MB per 32 C1 frames): spread it over the cores
        list(self._pool.map(pack, range(len(frames))))
        if len(frames) < B:
            for k in self.input_keys:
                host[k][len(frames):] = 0   # unused slots: empty frames (no features -> no work after the remap)

    def _predict(self, i0: int, chain: bool, token: int):
        """Reference slots for the pairs i0.. of the batch and what each assumes: ("key", token) = the keyframe as of now
        (slot 0), ("chain", j) = chunk[j - 1] will be the keyframe when frame j is resolved (slot j)."""
        B = self.cfg.batch
        refs, assume = [-1] * i0, [None] * i0
        for j in range(i0, B):
            if chain and j > i0:
                refs.append(j)
                assume.append(("chain", j))
            else:
                refs.append(0)
                assume.append(("key", token))
        return refs, assume

    def _h2d(self, s: int):
        for k in self.input_keys:
            self._dev[s][k].copy_(self._pinned[s][k], non_blocking=True)

    def _read(self):
        buf = self.fe.buffers()
        torch.cuda.synchronize(self.ctx.device)
        return (buf["pose"].cpu().numpy().astype(np.float64), buf["stats"].cpu().numpy(), buf["n"].cpu().numpy())

    def run(self, frames: Iterable[dict], frame_ids: Optional[Sequence[int]] = None, est_poses_file=None,
            keyframe_ids_file=None) -> VOResult:
        frames = list(frames)
        ids = list(range(len(frames))) if frame_ids is None else list(frame_ids)
        B = self.cfg.batch
        state = TrackingState(self.policy, self.number_of_cams, self.units_to_m)
        res = state.result
        self.fe.reset()
        nxt = 0                                   # next frame to resolve
        cur = 0                                   # staging set of the batch being resolved
        chain = False                             # predict "every frame becomes a keyframe" for the next batch
        packed = self._prefetch.submit(self._pack, frames[:B], cur)
        while nxt < len(frames) and res.status == "ok":
            chunk = frames[nxt:nxt + B]
            packed.result()
            self._h2d(cur)
            if nxt + B < len(frames):             # pack the next batch meanwhile
                packed = self._prefetch.submit(self._pack, frames[nxt + B:nxt + 2 * B], 1 - cur)
            first_batch = nxt == 0
            # Slot i+1 holds chunk[i]; slot 0 holds the current keyframe.  Which frame a pair is tracked against is a
            # PREDICTION of the keyframe decisions still to come: "no new keyframe" (reference = slot 0) or, when keyframes
            # have been frequent, "the previous frame becomes the keyframe" (reference = slot i, the chain).  A pair whose
            # prediction turns out wrong is re-tracked (stage B only) once the host knows better.  In the very first batch
            # frame 0 IS the first keyframe (create_keyframe starts True, pose_est_tools.py:1406).
            token, last_key = 0, -2                # keyframes created in this batch; chunk index of the newest one
            if first_batch:
                refs, assume = [-1] + [1] * (B - 1), [None] + [("key", 0)] * (B - 1)
            else:
                refs, assume = self._predict(0, chain, token)
            self.fe.set_ref_slots(refs)
            self._step(*[self._dev[cur][k] for k in self.input_keys])
            res.device_steps += 1
            pose, stats, n_slots = self._read()
            i = 0
            if first_batch:
                state.first_frame(ids[0], int(n_slots[1]))
                self.fe.promote(1)
                i = 1
            n_keys = 0
            while i < len(chunk):
                if assume[i] != ("key", token) and assume[i] != ("chain", last_key + 1):
                    refs, assume = self._predict(i, chain, token)
                    self.fe.set_ref_slots(refs)
                    self.fe.retrack()
                    res.device_retracks += 1
                    pose, stats, n_slots = self._read()
                n_corr, inliers, best = int(stats[i, 1]), int(stats[i, 2]), int(stats[i, 3])
                if n_corr < self.min_correspondences or best < 0:
                    res.status = f"tracking failed at frame {ids[nxt + i]}: {n_corr} point correspondences"
                    break
                if state.tracked_frame(ids[nxt + i], pose[i], inliers, int(n_slots[i + 1])):
                    self.fe.promote(i + 1)         # chunk[i] is the keyframe now
                    token, last_key, n_keys = token + 1, i, n_keys + 1
                i += 1
            chain = 2 * n_keys >= len(chunk)       # next batch: chain the pairs when keyframes were the rule
            nxt += len(chunk)
            cur = 1 - cur
        packed.result()                           # a batch packed ahead of a tracking failure is simply dropped
        if est_poses_file is not None:
            for fid, T in zip(res.frame_ids, res.poses_wrt_S):
                print(tum_line(fid, T), file=est_poses_file)
        if keyframe_ids_file is not None:
            for k in res.keyframe_ids:
                print(k, file=keyframe_ids_file)
        return res
