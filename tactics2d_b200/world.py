"""BatchedWorld: N scenarios x M participants of structure-of-arrays state in HBM.

This is the object behind the reference-shaped facades (``physics``, ``traffic``, ``envs``): it
owns the fp32 SoA tensors, the C-ABI context, and forwards ``step`` / ``check_events`` / ``reset``
to the sm_100a kernels.  PyTorch is only the device-memory container (``tensor.data_ptr()``) and
the stream provider; there is no eager/CPU implementation behind it.

Replaces the per-object loop of the reference tick: ``ScenarioManager.update`` ->
``physics_model.step`` -> ``agent.add_state`` -> ``check_status`` (envs/parking.py:352-392).
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .types import MODEL_DRIFT, TYPE_INACTIVE, TypeTable

CFG_ANY_PARTICIPANT = 1
CFG_STEER_FIRST = 2

F_DYNAMIC, F_STATIC, F_OUTBOUND = 1, 2, 4


@dataclass
class StepResult:
    """Device tensors written by one ``step`` (views of buffers owned by the world)."""

    flags: torch.Tensor        # uint8 [N, M]: bit0 dynamic collision, bit1 static collision, bit2 out of bound
    hit_index: torch.Tensor    # int16 [N, M]: lowest colliding participant index or -1
    hit_segment: torch.Tensor  # int16 [N, M]: lowest colliding map segment index or -1
    status: torch.Tensor       # uint8 [N]: ScenarioStatus
    done: torch.Tensor         # uint8 [N]
    iou: Optional[torch.Tensor] = None   # fp32 [N]: IoU(ego pose, target area) when a goal is set (Arrival.update)


@dataclass
class EnvResult:
    """Device tensors written by ``env_epilogue`` (views of buffers owned by the world, overwritten by the next call)."""

    reward: torch.Tensor          # fp32 [N]
    terminated: torch.Tensor      # bool [N]
    truncated: torch.Tensor       # bool [N]
    done: torch.Tensor            # uint8 [N] = terminated | truncated (the mask ``reset`` takes)
    traffic_status: torch.Tensor  # uint8 [N, M] TrafficStatus codes


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


class BatchedWorld:
    def __init__(self, n_scenarios: int, m_participants: int, type_table: TypeTable, device="cuda:0",
                 interval: int = 100, delta_t: int = 5, max_step: Optional[int] = None,
                 any_participant: bool = False, steer_first: bool = False):
        if not torch.cuda.is_available():
            raise RuntimeError("tactics2d_b200 needs a CUDA device: the batched tick only exists as sm_100a kernels")
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BatchedWorld lives on a CUDA device")
        self.N, self.M = int(n_scenarios), int(m_participants)
        self.type_table = type_table
        self.interval, self.delta_t = int(interval), int(delta_t)
        self.max_step = int(max_step) if max_step else 0
        self.flags_cfg = (CFG_ANY_PARTICIPANT if any_participant else 0) | (CFG_STEER_FIRST if steer_first else 0)
        self._ctx = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.dev_index = dev_index
        cfg = _lib.Config(self.interval, self.delta_t, self.max_step, self.flags_cfg)
        _lib.check(self.lib.t2d_create(C.byref(self._ctx), dev_index, self.N, self.M, C.byref(cfg)))
        arr = type_table.to_c_array()
        _lib.check(self.lib.t2d_set_type_table(self._ctx, arr, len(type_table)))

        f = dict(dtype=torch.float32, device=self.device)
        shape = (self.N, self.M)
        self.x = torch.zeros(shape, **f)
        self.y = torch.zeros(shape, **f)
        self.heading = torch.zeros(shape, **f)
        self.speed = torch.zeros(shape, **f)
        self.vx = torch.zeros(shape, **f)
        self.vy = torch.zeros(shape, **f)
        self.type_id = torch.full(shape, TYPE_INACTIVE, dtype=torch.uint8, device=self.device)
        self.step_count = torch.zeros(self.N, dtype=torch.int32, device=self.device)
        self.frame = 0  # ms; State.frame advances by `interval` per step (single_track_kinematics.py:166)
        self._out = StepResult(
            flags=torch.zeros(shape, dtype=torch.uint8, device=self.device),
            hit_index=torch.full(shape, -1, dtype=torch.int16, device=self.device),
            hit_segment=torch.full(shape, -1, dtype=torch.int16, device=self.device),
            status=torch.ones(self.N, dtype=torch.uint8, device=self.device),
            done=torch.zeros(self.N, dtype=torch.uint8, device=self.device))
        self._bind()
        # SingleTrackDrift participants carry their wheel speeds (single_track_drift.py:467-499)
        self.omega_front = self.omega_rear = None
        if any(r.model == MODEL_DRIFT for r in type_table.rows):
            self.omega_front = torch.zeros(shape, **f)
            self.omega_rear = torch.zeros(shape, **f)
            _lib.check(self.lib.t2d_bind_wheel_state(self._ctx, _ptr(self.omega_front), _ptr(self.omega_rear)))
        self.segments = None
        self.poly_start = None
        self.tiles, self.tile_id = None, None
        self.bounds = None
        self._goal = None

    # ------------------------------------------------------------------ plumbing
    def _bind(self):
        _lib.check(self.lib.t2d_bind_state(self._ctx, _ptr(self.x), _ptr(self.y), _ptr(self.heading), _ptr(self.speed),
                                           _ptr(self.vx), _ptr(self.vy), _ptr(self.type_id), _ptr(self.step_count)))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.t2d_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ configuration
    def set_config(self, interval=None, delta_t=None, max_step=None):
        if interval is not None:
            self.interval = int(interval)
        if delta_t is not None:
            self.delta_t = int(delta_t)
        if max_step is not None:
            self.max_step = int(max_step)
        cfg = _lib.Config(self.interval, self.delta_t, self.max_step, self.flags_cfg)
        _lib.check(self.lib.t2d_set_config(self._ctx, C.byref(cfg)))

    def set_map(self, segments=None, bounds: Optional[Sequence[float]] = None, cell_size: float = 0.0, poly_start=None):
        """Static geometry of the scenario (shared by all N scenarios).

        ``segments``: array [S, 4] of (x1, y1, x2, y2) collidable pieces in list order - what
        ``StaticCollision.reset(static_objects)`` receives (collision.py:45-46), flattened;
        ``bounds``: (xmin, xmax, ymin, ymax) as ``Map.boundary`` / ``OutBound.reset`` take it
        (out_bound.py:50-65), or None;
        ``poly_start``: int array [P + 1] marking the segments that close up to ``Area`` polygons (ring p = segments
        [poly_start[p], poly_start[p + 1])): a pose inside a polygon collides with it even when it touches no edge, and
        ``hit_segment`` then names the first object hit by its first segment (see :func:`polygons_to_segments`)."""
        seg = None if segments is None else np.ascontiguousarray(np.asarray(segments, dtype=np.float32).reshape(-1, 4))
        n_seg = 0 if seg is None else seg.shape[0]
        b = None if bounds is None else np.ascontiguousarray(np.asarray(bounds, dtype=np.float32))
        ps = None if poly_start is None else np.ascontiguousarray(np.asarray(poly_start, dtype=np.int32))
        n_poly = 0 if ps is None else len(ps) - 1
        _lib.check(self.lib.t2d_set_map_polygons(
            self._ctx, C.c_void_p(0 if n_seg == 0 else seg.ctypes.data), n_seg, C.c_void_p(0 if n_poly <= 0 else ps.ctypes.data),
            max(0, n_poly), C.c_void_p(0 if b is None else b.ctypes.data), float(cell_size)))
        self.segments = seg
        self.poly_start = ps
        self.bounds = None if b is None else tuple(float(v) for v in b)
        self.tiles, self.tile_id = None, None

    def set_map_table(self, tiles, tile_id, cell_size: float = 0.0):
        """A different map per scenario: ``tiles`` is a list of dicts ``{"segments": [S, 4], "bounds": (4,) or None,
        "poly_start": [P + 1] or None}`` (what ``_ParkingScenarioManager.reset`` builds per episode - the lot's wall and
        obstacle Areas and ``map_.boundary``, envs/parking.py:397-441 - or the reference's ``data/*_map`` files, one tile
        each: ``map.polygons_to_segments(map.load_areas(name, subtypes), [lines])``), ``tile_id`` an integer array [N]: the tile of every scenario.  The ids live in ``self.tile_id`` (uint16
        device tensor) and may be rewritten between ticks."""
        keep, rows = [], (_lib.MapTileC * len(tiles))()
        for i, t in enumerate(tiles):
            seg = t.get("segments")
            seg = None if seg is None or len(seg) == 0 else np.ascontiguousarray(np.asarray(seg, dtype=np.float32).reshape(-1, 4))
            b = t.get("bounds")
            b = None if b is None else np.ascontiguousarray(np.asarray(b, dtype=np.float32))
            ps = t.get("poly_start")
            ps = None if ps is None or len(ps) < 2 else np.ascontiguousarray(np.asarray(ps, dtype=np.int32))
            keep.append((seg, b, ps))
            rows[i].segments = None if seg is None else seg.ctypes.data
            rows[i].n_seg = 0 if seg is None else seg.shape[0]
            rows[i].poly_start = None if ps is None else ps.ctypes.data
            rows[i].n_poly = 0 if ps is None else len(ps) - 1
            rows[i].bounds = None if b is None else b.ctypes.data
        tid = torch.as_tensor(np.asarray(tile_id) if not torch.is_tensor(tile_id) else tile_id).to(torch.int64)
        if tid.numel() != self.N or int(tid.min()) < 0 or int(tid.max()) >= len(tiles):
            raise ValueError(f"tile_id must hold {self.N} indices into the {len(tiles)} tiles")
        tid = tid.to(torch.int16).to(self.device).contiguous()   # (bit pattern of uint16 for ids < 32768)
        # a rejected table leaves the previous map, and the ids it reads, in force: replace self.tile_id only on success
        _lib.check(self.lib.t2d_set_map_table(self._ctx, rows, len(tiles), _ptr(tid), float(cell_size)))
        self.tile_id = tid
        self.tiles = [dict(segments=k[0], bounds=None if k[1] is None else tuple(float(v) for v in k[1]), poly_start=k[2]) for k in keep]
        self.segments, self.poly_start, self.bounds = None, None, None

    def set_goal(self, target=None, arrival_threshold: float = 0.95, no_action_max_step: int = 100):
        """Target area per scenario for the ego (participant 0): array [N, 5] = (cx, cy, heading, half_len, half_wid),
        or None to disable.  Enables ``Arrival`` (IoU >= threshold -> COMPLETED, arrival.py:32-47) and ``NoAction``
        (IoU with the previous pose > 0.999 for more than ``no_action_max_step`` ticks, no_action.py:32-53) inside
        ``step``; ``StepResult.iou`` then holds the ego/target IoU."""
        if target is None:
            self._goal = None
            self._out.iou = None
            _lib.check(self.lib.t2d_set_goal(self._ctx, _ptr(None), 0.95, 0, _ptr(None), _ptr(None), _ptr(None)))
            return
        t = torch.as_tensor(np.asarray(target, dtype=np.float32) if not torch.is_tensor(target) else target)
        t = t.to(device=self.device, dtype=torch.float32).reshape(self.N, 5).contiguous()
        self._goal = dict(target=t, iou=torch.zeros(self.N, dtype=torch.float32, device=self.device),
                          last_pose=torch.zeros((self.N, 4), dtype=torch.float32, device=self.device),
                          count=torch.zeros(self.N, dtype=torch.int32, device=self.device))
        self._out.iou = self._goal["iou"]
        g = self._goal
        _lib.check(self.lib.t2d_set_goal(self._ctx, _ptr(g["target"]), float(arrival_threshold), int(no_action_max_step),
                                         _ptr(g["iou"]), _ptr(g["last_pose"]), _ptr(g["count"])))

    # ------------------------------------------------------------------ NPC controllers
    def set_paths(self, paths):
        """Pure-pursuit waypoint polylines: a list of ``[V_p, 2]`` arrays (the ``waypoints`` of
        ``PurePursuitController.step``, pure_pursuit_controller.py:76); ``path_id`` of ``set_controllers`` indexes it."""
        paths = [np.ascontiguousarray(np.asarray(p, dtype=np.float32).reshape(-1, 2)) for p in paths]
        self.paths = paths
        if not paths:
            _lib.check(self.lib.t2d_set_paths(self._ctx, _ptr(None), _ptr(None), 0))
            return
        xy = np.ascontiguousarray(np.concatenate(paths, 0))
        off = np.zeros(len(paths) + 1, np.int32)
        off[1:] = np.cumsum([len(p) for p in paths])
        _lib.check(self.lib.t2d_set_paths(self._ctx, C.c_void_p(xy.ctypes.data), C.c_void_p(off.ctypes.data), len(paths)))

    def set_controllers(self, controllers, ctrl_id, lead_index=None, path_id=None, last_accel=None):
        """Hand the non-ego agents to on-device controllers.  ``controllers``: list of ``tactics2d_b200.controller``
        objects (or ``ControllerParamsC`` rows); ``ctrl_id`` [N, M] uint8: the participant's row, 255 for "action comes
        from the caller"; ``lead_index`` [N, M] int16: its leading vehicle (``leading_state`` / ``front_state``), -1 for
        none; ``path_id`` [N, M] int16: its pure-pursuit path (``set_paths``), -1 for none; ``last_accel`` [N, M]:
        ``State.accel`` of the previous tick (default zeros).  ``None`` for ``controllers`` removes them."""
        if controllers is None:
            self._ctrl = None
            _lib.check(self.lib.t2d_set_controllers(self._ctx, _ptr(None), 0, _ptr(None), _ptr(None), _ptr(None), _ptr(None)))
            return
        rows = [c if isinstance(c, _lib.ControllerParamsC) else c.params() for c in controllers]
        arr = (_lib.ControllerParamsC * len(rows))(*rows)

        def dev(a, dtype, fill):
            if a is None:
                return None
            t = a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(np.asarray(a)))
            return t.to(device=self.device, dtype=dtype).reshape(self.N, self.M).contiguous()

        cid = dev(ctrl_id, torch.uint8, 255)
        lead = dev(lead_index, torch.int16, -1)
        pid = dev(path_id, torch.int16, -1)
        la = dev(last_accel, torch.float32, 0.0)
        if la is None:
            la = torch.zeros((self.N, self.M), dtype=torch.float32, device=self.device)
        self._ctrl = dict(rows=arr, ctrl_id=cid, lead_index=lead, path_id=pid, last_accel=la)
        _lib.check(self.lib.t2d_set_controllers(self._ctx, arr, len(rows), _ptr(cid), _ptr(lead), _ptr(pid), _ptr(la)))

    @property
    def last_accel(self) -> Optional[torch.Tensor]:
        c = getattr(self, "_ctrl", None)
        return None if c is None else c["last_accel"]

    def control(self, action: torch.Tensor) -> torch.Tensor:
        """Fill the rows of ``action`` [N, M, 2] that belong to controlled participants (IN PLACE; the other rows keep
        the caller's values) and refresh ``last_accel`` - ``ControllerBase.step`` of every NPC in one launch.  Call it
        after writing the external (ego) actions and before ``step``."""
        if action.device != self.device or action.dtype != torch.float32:
            raise ValueError("action must be an fp32 tensor on the world's device")
        if tuple(action.shape) != (self.N, self.M, 2) or not action.is_contiguous():
            raise ValueError(f"action must be contiguous [{self.N}, {self.M}, 2]")
        _lib.check(self.lib.t2d_control(self._ctx, _ptr(action), self._stream()))
        return action

    # ------------------------------------------------------------------ state
    def set_wheel_state(self, omega_front, omega_rear):
        """Wheel angular speeds [N, M] of the SingleTrackDrift participants (``omega_wf`` / ``omega_wr``)."""
        if self.omega_front is None:
            raise ValueError("the type table holds no SingleTrackDrift row")
        for dst, src in ((self.omega_front, omega_front), (self.omega_rear, omega_rear)):
            dst.copy_(torch.as_tensor(np.asarray(src) if not torch.is_tensor(src) else src).to(dst.dtype).reshape(dst.shape))

    def set_state(self, x, y, heading, speed=None, vx=None, vy=None, type_id=None):
        """Copy host or device arrays [N, M] into the SoA state.  Missing ``vx, vy`` are derived as
        ``State.velocity`` does (state.py:160-165); missing ``speed`` as ``State.speed`` (:143-146)."""
        def put(dst, src):
            dst.copy_(torch.as_tensor(np.asarray(src) if not torch.is_tensor(src) else src).to(dst.dtype).reshape(dst.shape))

        put(self.x, x); put(self.y, y); put(self.heading, heading)
        if speed is None and (vx is None or vy is None):
            raise ValueError("give speed, or vx and vy")
        if vx is not None and vy is not None:
            put(self.vx, vx); put(self.vy, vy)
        if speed is not None:
            put(self.speed, speed)
        else:
            self.speed.copy_(torch.sqrt(self.vx * self.vx + self.vy * self.vy))
        if vx is None or vy is None:
            self.vx.copy_(self.speed * torch.cos(self.heading))
            self.vy.copy_(self.speed * torch.sin(self.heading))
        if type_id is not None:
            put(self.type_id, type_id)

    def state_numpy(self) -> dict:
        out = {k: getattr(self, k).detach().cpu().numpy() for k in ("x", "y", "heading", "speed", "vx", "vy")}
        if self.omega_front is not None:
            out["omega_wf"] = self.omega_front.detach().cpu().numpy()
            out["omega_wr"] = self.omega_rear.detach().cpu().numpy()
        return out

    # ------------------------------------------------------------------ the hot path
    def step(self, action: torch.Tensor) -> StepResult:
        """One tick.  ``action``: fp32 device tensor [N, M, 2] = (accel, steer) per bicycle
        (``(steer, accel)`` when built with ``steer_first``), (ax, ay) per point mass."""
        if action.device != self.device or action.dtype != torch.float32:
            raise ValueError("action must be an fp32 tensor on the world's device")
        if tuple(action.shape) != (self.N, self.M, 2) or not action.is_contiguous():
            raise ValueError(f"action must be contiguous [{self.N}, {self.M}, 2]")
        o = self._out
        _lib.check(self.lib.t2d_step(self._ctx, _ptr(action), _ptr(o.flags), _ptr(o.hit_index), _ptr(o.hit_segment),
                                     _ptr(o.status), _ptr(o.done), self._stream()))
        self.frame += self.interval
        return o

    @property
    def result(self) -> StepResult:
        """The device-side output arrays of the last ``step`` / ``step_host`` / ``check_events``."""
        return self._out

    def step_host(self, action):
        """One tick for a host-side caller: ``action`` is a float32 ``[N, M, 2]`` NumPy array or CPU tensor (pinned
        memory avoids the driver's staging copy).  Returns ``(done, status)`` as uint8 NumPy arrays [N], valid on
        return; the per-participant flags / hit indices stay on the device in ``self.result`` (whose ``status`` /
        ``done`` tensors this call does not touch).  The copies are
        inside the call (``t2d_step_host``): chunked host->device copy overlapped with the kernel, one
        device->host read-back, one stream synchronisation."""
        a = action if isinstance(action, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(action, dtype=np.float32))
        if a.device.type != "cpu" or a.dtype != torch.float32 or tuple(a.shape) != (self.N, self.M, 2) or not a.is_contiguous():
            raise ValueError(f"action must be a contiguous float32 host array [{self.N}, {self.M}, 2]")
        hb = getattr(self, "_host_out", None)
        if hb is None:
            hb = self._host_out = (np.empty(self.N, np.uint8), np.empty(self.N, np.uint8))
        o = self._out
        _lib.check(self.lib.t2d_step_host(self._ctx, a.data_ptr(), _ptr(o.flags), _ptr(o.hit_index), _ptr(o.hit_segment),
                                          hb[1].ctypes.data, hb[0].ctypes.data, self._stream()))
        self.frame += self.interval
        return hb[0], hb[1]

    # ------------------------------------------------------------------ env layer
    def set_ego_action(self, ego_action: Optional[torch.Tensor]):
        """Bind the ego's action array: fp32 device tensor [N, 2] (or None to unbind).  While bound, ``control`` and
        ``step`` take the action of participant 0 of every scenario from it - the reference env's single action
        (envs/parking.py:219-239) - instead of row 0 of the full action array."""
        if ego_action is not None:
            if (ego_action.device != self.device or ego_action.dtype != torch.float32 or tuple(ego_action.shape) != (self.N, 2)
                    or not ego_action.is_contiguous()):
                raise ValueError(f"ego_action must be a contiguous fp32 [{self.N}, 2] tensor on {self.device}")
        self._ego_action = ego_action   # keeps the tensor alive while the library holds its pointer
        _lib.check(self.lib.t2d_set_ego_action(self._ctx, _ptr(ego_action)))

    def step_host_ego(self, ego_action, action: Optional[torch.Tensor] = None):
        """One tick for a host-side policy that drives only the ego: ``ego_action`` is a float32 ``[N, 2]`` NumPy array
        or CPU tensor; the other participants take the rows of the DEVICE array ``action`` [N, M, 2] (default: an
        internal zero array), which ``set_controllers`` fills on the device.  Per step 8 N bytes go up and 2 N come back
        (``t2d_step_host_ego``).  Returns ``(done, status)`` as uint8 NumPy arrays [N]."""
        a = ego_action if isinstance(ego_action, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(ego_action, dtype=np.float32))
        if a.device.type != "cpu" or a.dtype != torch.float32 or tuple(a.shape) != (self.N, 2) or not a.is_contiguous():
            raise ValueError(f"ego_action must be a contiguous float32 host array [{self.N}, 2]")
        if action is None:
            action = getattr(self, "_npc_action", None)
            if action is None:
                action = self._npc_action = torch.zeros((self.N, self.M, 2), dtype=torch.float32, device=self.device)
        elif action.device != self.device or action.dtype != torch.float32 or tuple(action.shape) != (self.N, self.M, 2) \
                or not action.is_contiguous():
            raise ValueError(f"action must be contiguous fp32 [{self.N}, {self.M}, 2] on {self.device}")
        hb = getattr(self, "_host_out", None)
        if hb is None:
            hb = self._host_out = (np.empty(self.N, np.uint8), np.empty(self.N, np.uint8))
        o = self._out
        _lib.check(self.lib.t2d_step_host_ego(self._ctx, a.data_ptr(), _ptr(action), _ptr(o.flags), _ptr(o.hit_index),
                                              _ptr(o.hit_segment), hb[1].ctypes.data, hb[0].ctypes.data, self._stream()))
        self.frame += self.interval
        return hb[0], hb[1]

    def set_prefetch(self, mode: int):
        """Tuning knob of the tick (``t2d_set_prefetch``), no effect on results: 1 / 0 = ask L2 for the next inputs early or
        not, -1 = the library's policy (on unless a peer-memory done exchange is alive)."""
        _lib.check(self.lib.t2d_set_prefetch(self._ctx, int(mode)))

    def env_epilogue(self, reset_trackers_on_done: bool = True) -> "EnvResult":
        """Reward, terminated, truncated, done and the per-participant TrafficStatus of the last tick in ONE launch
        (``t2d_env_epilogue``: ParkingEnv.step after check_status, envs/parking.py:240-256 and _get_reward :148-190)."""
        e = getattr(self, "_env", None)
        if e is None:
            u8 = dict(dtype=torch.uint8, device=self.device)
            e = self._env = dict(
                reward=torch.zeros(self.N, dtype=torch.float32, device=self.device),
                terminated=torch.zeros(self.N, dtype=torch.bool, device=self.device),
                truncated=torch.zeros(self.N, dtype=torch.bool, device=self.device),
                done=torch.zeros(self.N, **u8), traffic=torch.ones((self.N, self.M), **u8),
                max_iou=torch.full((self.N,), -float("inf"), dtype=torch.float32, device=self.device),
                min_dist=torch.full((self.N,), float("inf"), dtype=torch.float32, device=self.device))
        goal = self._goal is not None
        o = self._out
        _lib.check(self.lib.t2d_env_epilogue(self._ctx, _ptr(o.flags), _ptr(o.status), _ptr(e["reward"]), _ptr(e["terminated"]),
                                             _ptr(e["truncated"]), _ptr(e["traffic"]), _ptr(e["done"]),
                                             _ptr(e["max_iou"] if goal else None), _ptr(e["min_dist"] if goal else None),
                                             1 if reset_trackers_on_done else 0, self._stream()))
        return EnvResult(e["reward"], e["terminated"], e["truncated"], e["done"], e["traffic"])

    def reset_env_trackers(self):
        """``ParkingEnv.reset``: forget the best IoU / distance of the previous episodes (parking.py:276-277)."""
        e = getattr(self, "_env", None)
        if e is not None:
            e["max_iou"].fill_(-float("inf"))
            e["min_dist"].fill_(float("inf"))

    def check_events(self) -> StepResult:
        """The detectors on the current poses, no physics (``EventBase.update``)."""
        o = self._out
        _lib.check(self.lib.t2d_check_events(self._ctx, _ptr(o.flags), _ptr(o.hit_index), _ptr(o.hit_segment), self._stream()))
        return o

    def lidar_scan(self, n_beams: int = 500, max_range: float = 12.0) -> torch.Tensor:
        """Single-line lidar of every scenario's ego (``SingleLineLidar._scan_obstacles``, sensor/lidar.py:128-221):
        fp32 [N, n_beams] distances, ``inf`` where nothing is hit within ``max_range``.  Defaults are the
        reference's (range 12 m, freq_detect / freq_scan = 5000 / 10 = 500 beams, lidar.py:35-50)."""
        key = (int(n_beams), float(max_range))
        cache = getattr(self, "_lidar", None)
        if cache is None or cache[0] != key:
            theta = np.linspace(0, 2 * np.pi, int(n_beams), endpoint=False)          # lidar.py:160
            cs = torch.from_numpy(np.stack([np.cos(theta), np.sin(theta)], 1)).to(self.device)   # float64, host trig
            scan = torch.empty((self.N, int(n_beams)), dtype=torch.float32, device=self.device)
            self._lidar = cache = (key, cs.contiguous(), scan)
        _lib.check(self.lib.t2d_lidar_scan(self._ctx, int(n_beams), float(max_range), _ptr(cache[1]), _ptr(cache[2]), self._stream()))
        return cache[2]

    def reset(self, mask: torch.Tensor, pool: dict, pool_index: Optional[torch.Tensor] = None):
        """Re-initialise the scenarios with ``mask[n] != 0`` from row ``pool_index[n]`` (default n)
        of the pool arrays ``x, y, heading, speed[, vx, vy]`` [P, M] (``ScenarioManager.reset``,
        parking.py:397-441; ``ParticipantBase.reset``, participant_base.py:236-246)."""
        px = pool["x"]
        n_pool = px.shape[0]
        cols = ["x", "y", "heading", "speed"] + [k for k in ("vx", "vy", "omega_wf", "omega_wr") if pool.get(k) is not None]
        for k in cols:
            t = pool[k]
            if t.device != self.device or t.dtype != torch.float32 or tuple(t.shape) != (n_pool, self.M) or not t.is_contiguous():
                raise ValueError(f"pool[{k!r}] must be a contiguous fp32 [{n_pool}, {self.M}] tensor on {self.device}")
        if (pool.get("vx") is None) != (pool.get("vy") is None):
            raise ValueError("give both pool['vx'] and pool['vy'], or neither")
        # mask / pool_index reach the kernel as raw pointers: a host tensor or a wrong length would be an illegal address
        if not torch.is_tensor(mask) or mask.numel() != self.N:
            raise ValueError(f"mask must be a tensor of {self.N} scenarios")
        mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        if pool_index is not None:
            if not torch.is_tensor(pool_index) or pool_index.numel() != self.N:
                raise ValueError(f"pool_index must be a tensor of {self.N} scenarios")
            pool_index = pool_index.to(device=self.device, dtype=torch.int32).contiguous()
        if pool_index is None and n_pool < self.N:
            raise ValueError("without pool_index the pool needs one row per scenario")
        if self.omega_front is not None:
            wf, wr = pool.get("omega_wf"), pool.get("omega_wr")
            if (wf is None) != (wr is None):
                raise ValueError("give both pool['omega_wf'] and pool['omega_wr'], or neither")
            _lib.check(self.lib.t2d_bind_reset_wheel_pool(self._ctx, _ptr(wf), _ptr(wr)))
        _lib.check(self.lib.t2d_reset(self._ctx, _ptr(mask), _ptr(pool_index), n_pool, _ptr(pool["x"]), _ptr(pool["y"]),
                                      _ptr(pool["heading"]), _ptr(pool["speed"]), _ptr(pool.get("vx")),
                                      _ptr(pool.get("vy")), self._stream()))
