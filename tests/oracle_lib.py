"""ctypes wrapper of the CPU oracle (oracle/wl_oracle.c).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ODIR = ROOT / "oracle"


def _ensure_built():
    subprocess.run(["make", "-C", str(ODIR), "libwl_oracle.so", "libwl_oracle_f64.so"], check=True, stdout=subprocess.DEVNULL)


def _load_native():
    """The -march=native build is compiled for the host that loads it, in a temporary directory (the tree may be
    read-only); the file is removed once it is mapped, so every process that loads it pays the few-second compile."""
    with tempfile.TemporaryDirectory(prefix="wl_oracle_native_") as d:
        subprocess.run(["make", "-C", str(ODIR), f"NATIVE_DIR={d}", f"{d}/libwl_oracle_native.so"], check=True, stdout=subprocess.DEVNULL)
        return _load(Path(d) / "libwl_oracle_native.so")


def _load(path):
    lib = C.CDLL(str(path))
    vp, i32, i64, u32, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64
    lib.wlo_create.restype = vp
    lib.wlo_create.argtypes = [vp, vp]
    lib.wlo_destroy.argtypes = [vp]
    lib.wlo_startup.argtypes = [vp]
    lib.wlo_reset.argtypes = [vp, vp, i32, i64]
    lib.wlo_step.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32]
    lib.wlo_observe.argtypes = [vp, vp, i64, i32]
    lib.wlo_curriculum.argtypes = [vp, i32, vp, vp, u32]
    lib.wlo_synth_actions.argtypes = [vp, vp, i64, i32]
    lib.wlo_export_state.argtypes = [vp, vp]
    lib.wlo_import_state.argtypes = [vp, vp]
    lib.wlo_get_weights.argtypes = [vp, vp]
    lib.wlo_set_weights.argtypes = [vp, vp]
    lib.wlo_get_log.argtypes = [vp, vp]
    lib.wlo_any_reset_last.argtypes = [vp]
    lib.wlo_detmath.argtypes = [i32, vp, vp, vp, i32]
    lib.wlo_philox.argtypes = [u64, u32, u32, u32, u32, vp, i32]
    lib.wlo_action_map.argtypes = [vp, vp, vp, vp, i32]
    lib.wlo_drift_terms.argtypes = [vp, vp, vp, vp, vp, vp, i32]
    lib.wlo_euler_xyz.argtypes = [vp, vp, i32]
    lib.wlo_drift_reset_pose.argtypes = [vp, vp, vp, vp, vp, i32]
    lib.wlo_elev_terms.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32]
    lib.wlo_dc_motor.argtypes = [vp, C.c_float, C.c_float, vp, vp, vp, i32]
    lib.wlo_camera.argtypes = [vp, vp, i64, vp]
    lib.wlo_camera_post.argtypes = [vp, vp, vp, vp, i32]
    lib.wlo_camera_render.argtypes = [vp, i32, vp]
    lib.wlo_config_describe.restype = C.c_char_p
    return lib


_libs = {}


def get_lib(kind="f32"):
    if kind not in _libs:
        if kind == "native":
            _libs[kind] = _load_native()
        else:
            _ensure_built()
            _libs[kind] = _load(ODIR / {"f32": "libwl_oracle.so", "f64": "libwl_oracle_f64.so"}[kind])
    return _libs[kind]


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


NUM_GROUPS = 16

_CFG_CLS = None


def config_struct():
    """ctypes mirror of wl_config built from the ORACLE's own field list (wlo_config_describe), so that the reference arm of
    bench.py can drive the oracle from a committed config blob without importing the product package."""
    global _CFG_CLS
    if _CFG_CLS is None:
        tags = {"i32": C.c_int32, "u64": C.c_uint64, "f32": C.c_float}
        fields, size = [], None
        for item in get_lib().wlo_config_describe().decode().split(";"):
            if not item:
                continue
            parts = item.split(":")
            if parts[0] == "sizeof":
                size = int(parts[1]); continue
            ct = tags[parts[1]]
            fields.append((parts[0], ct if int(parts[2]) == 1 else ct * int(parts[2])))
        _CFG_CLS = type("WloConfig", (C.Structure,), {"_fields_": fields})
        assert size is None or C.sizeof(_CFG_CLS) == size
    return _CFG_CLS


def cfg_from_blob(path, **overrides):
    """wl_config from a binary blob (python -m wheeledlab_b200.dump_config / tests/golden/cfg_blobs) + field overrides."""
    cls = config_struct()
    raw = Path(path).read_bytes()
    assert len(raw) == C.sizeof(cls), f"{path}: {len(raw)} bytes, wl_config is {C.sizeof(cls)} (stale blob? regenerate)"
    cfg = cls.from_buffer_copy(raw)
    for k, v in overrides.items():
        setattr(cfg, k, v)
    return cfg


class Oracle:
    """One oracle instance; mirrors the wl_* calls with host (numpy) buffers."""

    def __init__(self, cfg, heightfield=None, kind="f32", threads=1):
        self.lib = get_lib(kind)
        self.cfg = cfg
        self.n = int(cfg.num_envs)
        self.threads = threads
        self.obs_dim = {0: 14, 1: 689, 2: 8}[int(cfg.task)]
        if int(cfg.task) == 2 and int(cfg.vis_cam):
            self.obs_dim += int(cfg.vis_cam_w) * (int(cfg.vis_cam_h) - int(cfg.vis_cam_row0))
        if heightfield is None:
            hf = None
        elif int(cfg.task) == 2:
            hf = np.ascontiguousarray(heightfield)                      # raw aux bytes (visual)
        else:
            hf = np.ascontiguousarray(heightfield, dtype=np.float32)
        self._h = C.c_void_p(self.lib.wlo_create(C.byref(cfg), _p(hf)))

    def __del__(self):
        try:
            self.lib.wlo_destroy(self._h)
        except Exception:
            pass

    def startup(self):
        assert self.lib.wlo_startup(self._h) == 0

    def reset(self, env_ids, step_counter):
        if env_ids is None:
            rc = self.lib.wlo_reset(self._h, None, 0, step_counter)
        else:
            ids = np.ascontiguousarray(env_ids, dtype=np.int64)
            rc = self.lib.wlo_reset(self._h, _p(ids), len(ids), step_counter)
        assert rc == 0

    def step(self, action, step_counter):
        a = np.ascontiguousarray(action, dtype=np.float32)
        obs = np.empty((self.n, self.obs_dim), np.float32)
        rew = np.empty(self.n, np.float32)
        term = np.empty(self.n, np.uint8)
        trunc = np.empty(self.n, np.uint8)
        rc = self.lib.wlo_step(self._h, _p(a), _p(obs), _p(rew), _p(term), _p(trunc), step_counter, self.threads)
        assert rc == 0, rc
        return obs, rew, term, trunc

    def observe(self, step_counter, call_idx=0):
        obs = np.empty((self.n, self.obs_dim), np.float32)
        assert self.lib.wlo_observe(self._h, _p(obs), step_counter, call_idx) == 0
        return obs

    def curriculum(self, slots, increases, fire_mask):
        s = np.asarray(slots, np.int32)
        i = np.asarray(increases, np.float32)
        assert self.lib.wlo_curriculum(self._h, len(s), _p(s), _p(i), fire_mask) == 0

    def synth_actions(self, step_counter, dist=0):
        a = np.empty((self.n, 2), np.float32)
        assert self.lib.wlo_synth_actions(C.byref(self.cfg), _p(a), step_counter, dist) == 0
        return a

    def export_state(self):
        buf = np.zeros((NUM_GROUPS, self.n, 4), np.float32)
        self.lib.wlo_export_state(self._h, _p(buf))
        return buf

    def import_state(self, buf):
        b = np.ascontiguousarray(buf, dtype=np.float32)
        self.lib.wlo_import_state(self._h, _p(b))

    def weights(self):
        w = np.zeros(8, np.float32)
        self.lib.wlo_get_weights(self._h, _p(w))
        return w

    def set_weights(self, w):
        w = np.ascontiguousarray(w, np.float32)
        self.lib.wlo_set_weights(self._h, _p(w))

    def camera(self, step_counter, aug=None):
        """Camera term alone into a fresh [n, obs_dim] buffer (only the camera floats are written)."""
        obs = np.zeros((self.n, self.obs_dim), np.float32)
        a = None if aug is None else np.ascontiguousarray(aug, np.float32)
        assert self.lib.wlo_camera(self._h, _p(obs), step_counter, _p(a)) == 0
        return obs

    def camera_render(self, li):
        npix = self.obs_dim - 8
        out = np.zeros(npix, np.uint8)
        assert self.lib.wlo_camera_render(self._h, li, _p(out)) == 0
        return out

    def any_reset(self) -> bool:
        """>= 1 env reset in the most recent step (the log row itself persists over steps without a reset)."""
        return bool(self.lib.wlo_any_reset_last(self._h))

    def log(self):
        out = np.zeros(16, np.float64)
        self.lib.wlo_get_log(self._h, _p(out))
        return out


def detmath(op, x, x2=None, kind="f32"):
    lib = get_lib(kind)
    x = np.ascontiguousarray(x, np.float32)
    x2 = x if x2 is None else np.ascontiguousarray(x2, np.float32)
    out = np.empty_like(x)
    assert lib.wlo_detmath(op, _p(x), _p(x2), _p(out), x.size) == 0
    return out


def dc_motor(cfg, kd, effort_limit, target, omega):
    t = np.ascontiguousarray(target, np.float32); w = np.ascontiguousarray(omega, np.float32)
    out = np.empty_like(t)
    assert get_lib().wlo_dc_motor(C.byref(cfg), kd, effort_limit, _p(t), _p(w), _p(out), t.size) == 0
    return out


def camera_post(cfg, white, aug, kind="f32"):
    """camera_data_rgb_flattened[_aug] on white masks [n, rows*W] with explicit ColorJitter / blur parameters (9 floats)."""
    white = np.ascontiguousarray(white, np.uint8)
    out = np.empty(white.shape, np.float32)
    a = None if aug is None else np.ascontiguousarray(aug, np.float32)
    assert get_lib(kind).wlo_camera_post(C.byref(cfg), _p(white), _p(a), _p(out), white.shape[0]) == 0
    return out


def philox(seed, c0_base, c1, c2, c3, n):
    out = np.empty((n, 4), np.uint32)
    assert get_lib().wlo_philox(seed, c0_base, c1, c2, c3, _p(out), n) == 0
    return out


def action_map(cfg, action):
    a = np.ascontiguousarray(action, np.float32)
    n = a.shape[0]
    wheel = np.empty((n, 4), np.float32)
    steer = np.empty((n, 2), np.float32)
    rc = get_lib().wlo_action_map(C.byref(cfg), _p(a), _p(wheel), _p(steer), n)
    assert rc == 0, rc
    return wheel, steer


def drift_terms(cfg, root, steer, ep_len):
    root = np.ascontiguousarray(root, np.float32)
    steer = np.ascontiguousarray(steer, np.float32)
    ep = np.ascontiguousarray(ep_len, np.int32)
    n = root.shape[0]
    f = np.empty((n, 8), np.float32)
    oob = np.empty(n, np.uint8)
    assert get_lib().wlo_drift_terms(C.byref(cfg), _p(root), _p(steer), _p(ep), _p(f), _p(oob), n) == 0
    return f, oob


def euler_xyz(quat):
    q = np.ascontiguousarray(quat, np.float32)
    out = np.empty((q.shape[0], 3), np.float32)
    assert get_lib().wlo_euler_xyz(_p(q), _p(out), q.shape[0]) == 0
    return out


def drift_reset_pose(cfg, idx, u_xy, u_yaw):
    idx = np.ascontiguousarray(idx, np.int32)
    u_xy = np.ascontiguousarray(u_xy, np.float32)
    u_yaw = np.ascontiguousarray(u_yaw, np.float32)
    pose = np.empty((idx.shape[0], 7), np.float32)
    assert get_lib().wlo_drift_reset_pose(C.byref(cfg), _p(idx), _p(u_xy), _p(u_yaw), _p(pose), idx.shape[0]) == 0
    return pose


def elev_terms(cfg, root, cmdb, omega, action, ep_len):
    root = np.ascontiguousarray(root, np.float32); cmdb = np.ascontiguousarray(cmdb, np.float32)
    omega = np.ascontiguousarray(omega, np.float32); action = np.ascontiguousarray(action, np.float32)
    ep = np.ascontiguousarray(ep_len, np.int32)
    n = root.shape[0]
    f = np.empty((n, 8), np.float32); mask = np.empty(n, np.uint32); prop = np.empty((n, 13), np.float32)
    assert get_lib().wlo_elev_terms(C.byref(cfg), _p(root), _p(cmdb), _p(omega), _p(action), _p(ep), _p(f), _p(mask), _p(prop), n) == 0
    return f, mask, prop
