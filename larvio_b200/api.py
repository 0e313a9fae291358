"""ctypes binding of include/larvio_b200.h plus numpy-friendly wrappers.

Mirrors the reference's two classes for a batch of S sequences:
``Batch.process_images`` = ImageProcessor::processImage (image_processor.cpp:130-219),
``Batch.process_features`` = LarVio::processFeatures (larvio.cpp:363-461),
``Batch.step`` = the driver loop body (app/larvioMain.cpp:107-114).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Tuple

import numpy as np

from .config import Config, LvbConfig

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "liblarvio_b200.so")


class LarvioB200Error(RuntimeError):
    pass


def _load():
    if not os.path.exists(_LIB_PATH):
        raise LarvioB200Error(
            f"{_LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
            "There is no CPU fallback.")
    return C.CDLL(_LIB_PATH)


_lib = _load()


class LvbImu(C.Structure):
    _fields_ = [("t", C.c_double), ("gyro", C.c_double * 3), ("acc", C.c_double * 3)]


class LvbFeature(C.Structure):
    _fields_ = [("id", C.c_uint64), ("u", C.c_double), ("v", C.c_double), ("u_init", C.c_double),
                ("v_init", C.c_double), ("u_vel", C.c_double), ("v_vel", C.c_double),
                ("u_init_vel", C.c_double), ("v_init_vel", C.c_double)]


FEATURE_DTYPE = np.dtype([("id", np.uint64), ("u", np.float64), ("v", np.float64), ("u_init", np.float64),
                          ("v_init", np.float64), ("u_vel", np.float64), ("v_vel", np.float64),
                          ("u_init_vel", np.float64), ("v_init_vel", np.float64)])
IMU_DTYPE = np.dtype([("t", np.float64), ("gyro", np.float64, 3), ("acc", np.float64, 3)])

_vp = C.c_void_p
_lib.lvb_last_error.restype = C.c_char_p
_lib.lvb_launch_count.restype = C.c_longlong
_lib.lvb_launch_count.argtypes = [_vp]
_lib.lvb_create.argtypes = [C.POINTER(LvbConfig), C.c_int, C.c_int, C.POINTER(_vp)]
_lib.lvb_create_from_file.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(_vp)]
_lib.lvb_parse_config.argtypes = [C.c_char_p, C.POINTER(LvbConfig)]
_lib.lvb_destroy.argtypes = [_vp]
_lib.lvb_destroy.restype = None
_lib.lvb_feature_capacity.argtypes = [_vp]
_lib.lvb_n_seq.argtypes = [_vp]
_lib.lvb_synchronize.argtypes = [_vp]
_lib.lvb_profile_enable.argtypes = [_vp, C.c_int]
_lib.lvb_profile_reset.argtypes = [_vp]
_lib.lvb_get_stats.argtypes = [_vp, C.POINTER(C.c_ulonglong)]
_lib.lvb_get_stats.restype = C.c_int
_lib.lvb_debug_icore.argtypes = [_vp, C.c_int, C.POINTER(C.c_int)]
_lib.lvb_debug_icore.restype = C.c_int
_lib.lvb_profile_get.argtypes = [_vp, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.c_int]
for _name in ("lvbk_pyramid", "lvbk_pyramid_padded", "lvbk_lk", "lvbk_orb", "lvbk_detect", "lvbk_undistort", "lvbk_ransac",
              "lvb_process_images", "lvb_process_features", "lvb_step", "lvb_set_initial_state",
              "lvb_get_state", "lvb_get_states", "lvb_get_window", "lvb_get_covariance", "lvb_get_calibration", "lvb_get_points"):
    if hasattr(_lib, _name):
        getattr(_lib, _name).restype = C.c_int

LVB_PAD = 24          # pyramid level pad (lvb_internal.h)

EXPORTED_SYMBOLS = [
    "lvb_parse_config", "lvb_create", "lvb_create_from_file", "lvb_destroy", "lvb_last_error",
    "lvb_feature_capacity", "lvb_n_seq", "lvb_process_images", "lvb_process_features", "lvb_step",
    "lvb_synchronize", "lvb_set_initial_state", "lvb_get_state", "lvb_get_states", "lvb_get_window",
    "lvb_get_covariance", "lvb_get_calibration", "lvb_static_init_create", "lvb_static_init_destroy", "lvb_static_init_try", "lvbk_pyramid", "lvbk_pyramid_padded", "lvbk_lk", "lvbk_orb", "lvbk_detect", "lvbk_undistort",
    "lvbk_ransac", "lvb_launch_count", "lvb_profile_enable", "lvb_profile_reset", "lvb_profile_get", "lvb_get_stats", "lvb_debug_icore",
    "lvb_get_points", "lvbm_create", "lvbm_destroy", "lvbm_n_shards", "lvbm_set_initial_state", "lvbm_step", "lvbm_get_states",
    "lvbm_launch_count",
]


class MultiBatch:
    """lvbm_*: the batch sharded over several GPUs (or several shards of one GPU) inside one process."""

    def __init__(self, cfg, n_seq: int, gpu_ids):
        self.S = n_seq
        ids = (C.c_int * len(gpu_ids))(*gpu_ids)
        h = _vp()
        _lib.lvbm_create.restype = C.c_int; _lib.lvbm_step.restype = C.c_int; _lib.lvbm_get_states.restype = C.c_int
        _lib.lvbm_set_initial_state.restype = C.c_int; _lib.lvbm_launch_count.restype = C.c_longlong
        _lib.lvbm_launch_count.argtypes = [_vp]; _lib.lvbm_destroy.argtypes = [_vp]; _lib.lvbm_destroy.restype = None
        st = cfg.to_struct() if hasattr(cfg, "to_struct") else cfg
        _check(_lib.lvbm_create(C.byref(st), n_seq, ids, len(gpu_ids), C.byref(h)))
        self._h = h

    def set_initial_state(self, seq, t, q_xyzw, p, v, bg, ba):
        a = [np.ascontiguousarray(x, np.float64) for x in (q_xyzw, p, v, bg, ba)]
        _check(_lib.lvbm_set_initial_state(self._h, int(seq), C.c_double(float(t)), *[_p(x) for x in a]))

    def step(self, images, t_img, imu, n_imu):
        images = np.ascontiguousarray(images, np.uint8); t_img = np.ascontiguousarray(t_img, np.float64)
        pub = np.zeros(self.S, np.uint8)
        _check(_lib.lvbm_step(self._h, _p(images), _p(t_img), _p(imu), _p(n_imu), imu.shape[1], _p(pub)))
        return pub

    def get_states(self):
        out = np.zeros((self.S, 17))
        _check(_lib.lvbm_get_states(self._h, _p(out)))
        return out

    @property
    def launches(self):
        return int(_lib.lvbm_launch_count(self._h))

    def close(self):
        if self._h:
            _lib.lvbm_destroy(self._h); self._h = None


if hasattr(_lib, "lvb_static_init_create"):
    _lib.lvb_static_init_create.restype = C.c_void_p
    _lib.lvb_static_init_destroy.restype = None
    _lib.lvb_static_init_try.restype = C.c_int


def _check(rc: int):
    if rc != 0:
        raise LarvioB200Error(f"larvio_b200 error {rc}: {_lib.lvb_last_error().decode()}")


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(_vp)


def parse_config(path: str) -> LvbConfig:
    c = LvbConfig()
    _check(_lib.lvb_parse_config(path.encode(), C.byref(c)))
    return c


class StaticInitializer:
    """Host-side inclinometer initialiser of ONE sequence (StaticInitializer.cpp behind larvio.cpp:375-391); needs no GPU.
    try_init returns None until the scene was static for static_duration, then the start state for
    Batch.set_initial_state plus the number of IMU samples the caller erases from its buffer."""

    def __init__(self, cfg):
        st = cfg.to_struct() if hasattr(cfg, "to_struct") else cfg
        self._s = C.c_void_p(_lib.lvb_static_init_create(C.byref(st)))
        if not self._s:
            raise LarvioB200Error("lvb_static_init_create failed: " + _lib.lvb_last_error().decode())

    def try_init(self, feat: np.ndarray, t_msg: float, imu: np.ndarray):
        feat = np.ascontiguousarray(feat, FEATURE_DTYPE); imu = np.ascontiguousarray(imu, IMU_DTYPE)
        st = np.zeros(17); g = np.zeros(3); a = np.zeros(3); n = C.c_int()
        rc = _lib.lvb_static_init_try(self._s, _p(feat), len(feat), C.c_double(t_msg), _p(imu), len(imu), _p(st), _p(g), _p(a), C.byref(n))
        if rc < 0:
            _check(rc)
        if rc == 0:
            return None
        return dict(t=st[0], q=st[1:5].copy(), p=st[5:8].copy(), v=st[8:11].copy(), bg=st[11:14].copy(), ba=st[14:17].copy(),
                    gyro_old=g, acc_old=a, n_consumed=n.value)

    def close(self):
        if self._s:
            _lib.lvb_static_init_destroy(self._s); self._s = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Batch:
    """S independent (ImageProcessor, LarVio) pairs living on one GPU."""

    def __init__(self, cfg, n_seq: int = 1, device: int = 0):
        self._h = _vp()
        if isinstance(cfg, str):
            _check(_lib.lvb_create_from_file(cfg.encode(), n_seq, device, C.byref(self._h)))
        else:
            st = cfg.to_struct() if isinstance(cfg, Config) else cfg
            _check(_lib.lvb_create(C.byref(st), n_seq, device, C.byref(self._h)))
        self.S = n_seq
        self.cap = _lib.lvb_feature_capacity(self._h)

    def close(self):
        if self._h:
            _lib.lvb_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(_lib.lvb_launch_count(self._h))

    def profile(self, on: bool):
        _check(_lib.lvb_profile_enable(self._h, int(on)))

    def profile_reset(self):
        _check(_lib.lvb_profile_reset(self._h))

    def profile_get(self):
        cap = 128
        names = (C.c_char_p * cap)(); ms = (C.c_double * cap)(); cnt = (C.c_longlong * cap)()
        n = _lib.lvb_profile_get(self._h, names, ms, cnt, cap)
        return {names[i].decode(): (ms[i], int(cnt[i])) for i in range(min(n, cap))}

    def stats(self):
        out = (C.c_ulonglong * 16)()
        _check(_lib.lvb_get_stats(self._h, out))
        return [int(x) for x in out]

    def debug_icore(self, seq):
        out = (C.c_int * 32)()
        _check(_lib.lvb_debug_icore(self._h, seq, out))
        return [int(x) for x in out]

    def synchronize(self):
        _check(_lib.lvb_synchronize(self._h))

    # ---------------- stage-level entry points (parity tests) ----------------
    def k_pyramid(self, images: np.ndarray):
        images = np.ascontiguousarray(images, np.uint8)
        n, H, W = images.shape
        clahe = np.empty((n, H, W), np.uint8)
        l1 = np.empty((n, (H + 1) // 2, (W + 1) // 2), np.uint8)
        l2 = np.empty((n, (l1.shape[1] + 1) // 2, (l1.shape[2] + 1) // 2), np.uint8)
        blur = np.empty((n, H, W), np.uint8)
        _check(_lib.lvbk_pyramid(self._h, _p(images), n, _p(clahe), _p(l1), _p(l2), _p(blur)))
        return clahe, l1, l2, blur

    def k_pyramid_padded(self, images: np.ndarray, level: int):
        """Level `level` of the pyramid with its REFLECT_101 pad of LVB_PAD pixels: [n][h + 2 LVB_PAD][w + 2 LVB_PAD]."""
        images = np.ascontiguousarray(images, np.uint8)
        n, h, w = images.shape
        for _ in range(level):
            h, w = (h + 1) // 2, (w + 1) // 2
        out = np.empty((n, h + 2 * LVB_PAD, w + 2 * LVB_PAD), np.uint8)
        _check(_lib.lvbk_pyramid_padded(self._h, _p(images), n, int(level), _p(out)))
        return out

    def k_lk(self, prev: np.ndarray, nxt: np.ndarray, prev_pts: np.ndarray, init_pts: np.ndarray):
        prev = np.ascontiguousarray(prev, np.uint8); nxt = np.ascontiguousarray(nxt, np.uint8)
        n = prev.shape[0]
        pp = np.ascontiguousarray(prev_pts, np.float32).reshape(n, -1, 2)
        m = pp.shape[1]
        out = np.ascontiguousarray(init_pts, np.float32).reshape(n, m, 2).copy()
        st = np.zeros((n, m), np.uint8)
        _check(_lib.lvbk_lk(self._h, _p(prev), _p(nxt), n, m, _p(pp), _p(out), _p(st)))
        return out, st

    def k_orb(self, images: np.ndarray, pts: np.ndarray):
        images = np.ascontiguousarray(images, np.uint8)
        n = images.shape[0]
        pp = np.ascontiguousarray(pts, np.float32).reshape(n, -1, 2)
        m = pp.shape[1]
        ang = np.zeros((n, m), np.float32)
        desc = np.zeros((n, m, 32), np.uint8)
        _check(_lib.lvbk_orb(self._h, _p(images), n, m, _p(pp), _p(ang), _p(desc)))
        return ang, desc

    def k_detect(self, images: np.ndarray, masks: Optional[np.ndarray], want, return_eig=False):
        images = np.ascontiguousarray(images, np.uint8)
        n, H, W = images.shape
        if masks is not None:
            masks = np.ascontiguousarray(masks, np.uint8)
        want = np.ascontiguousarray(np.broadcast_to(np.asarray(want, np.int32), (n,)))
        out = np.zeros((n, self.cap, 2), np.float32)
        cnt = np.zeros(n, np.int32)
        eig = np.zeros((n, H, W), np.float32) if return_eig else None
        _check(_lib.lvbk_detect(self._h, _p(images), _p(masks), n, _p(want), _p(out), _p(cnt), _p(eig)))
        pts = [out[i, :cnt[i]].copy() for i in range(n)]
        return (pts, eig) if return_eig else pts

    def k_undistort(self, pts: np.ndarray, to_pixels: bool):
        pp = np.ascontiguousarray(pts, np.float32).reshape(-1, 2)
        out = np.zeros_like(pp)
        _check(_lib.lvbk_undistort(self._h, _p(pp), pp.shape[0], int(to_pixels), _p(out)))
        return out

    def k_ransac(self, p1: List[np.ndarray], p2: List[np.ndarray]):
        n = len(p1)
        m = np.array([len(a) for a in p1], np.int32)
        stride = int(max(1, m.max()))
        a = np.zeros((n, stride, 2), np.float32); b = np.zeros((n, stride, 2), np.float32)
        for i in range(n):
            a[i, :m[i]] = p1[i]; b[i, :m[i]] = p2[i]
        mask = np.zeros((n, stride), np.uint8)
        _check(_lib.lvbk_ransac(self._h, _p(a), _p(b), n, _p(m), stride, _p(mask)))
        return [mask[i, :m[i]].copy() for i in range(n)]

    # ---------------- the reference's call surface ----------------
    @staticmethod
    def pack_imu(rows_per_seq: List[np.ndarray], stride: Optional[int] = None):
        """rows [t,wx,wy,wz,ax,ay,az] per sequence -> (LvbImu[S][stride], n[S])."""
        S = len(rows_per_seq)
        stride = stride or max(1, max(len(r) for r in rows_per_seq))
        buf = np.zeros((S, stride), IMU_DTYPE)
        n = np.zeros(S, np.int32)
        for s, r in enumerate(rows_per_seq):
            k = len(r)
            n[s] = k
            if k:
                buf["t"][s, :k] = r[:, 0]; buf["gyro"][s, :k] = r[:, 1:4]; buf["acc"][s, :k] = r[:, 4:7]
        return buf, n

    def process_images(self, images: np.ndarray, t_img: np.ndarray, imu: np.ndarray, n_imu: np.ndarray):
        images = np.ascontiguousarray(images, np.uint8)
        t_img = np.ascontiguousarray(t_img, np.float64)
        feat = np.zeros((self.S, self.cap), FEATURE_DTYPE)
        out_n = np.zeros(self.S, np.int32)
        has = np.zeros(self.S, np.uint8)
        _check(_lib.lvb_process_images(self._h, _p(images), _p(t_img), _p(imu), _p(n_imu), imu.shape[1],
                                       _p(feat), _p(out_n), _p(has)))
        return feat, out_n, has

    def process_features(self, valid, t_msg, feat, n_feat, imu, n_imu):
        ok = np.zeros(self.S, np.uint8)
        valid = np.ascontiguousarray(valid, np.uint8)
        t_msg = np.ascontiguousarray(t_msg, np.float64)
        n_feat = np.ascontiguousarray(n_feat, np.int32)
        _check(_lib.lvb_process_features(self._h, _p(valid), _p(t_msg), _p(feat), _p(n_feat), feat.shape[1],
                                         _p(imu), _p(n_imu), imu.shape[1], _p(ok)))
        return ok

    def step(self, images, t_img, imu, n_imu, images_on_device: bool = False):
        pub = np.zeros(self.S, np.uint8)
        t_img = np.ascontiguousarray(t_img, np.float64)
        ptr = C.c_void_p(int(images)) if images_on_device else _p(np.ascontiguousarray(images, np.uint8))
        _check(_lib.lvb_step(self._h, ptr, int(images_on_device), _p(t_img), _p(imu), _p(n_imu),
                             imu.shape[1], _p(pub)))
        return pub

    def set_initial_state(self, seq, t, q_xyzw, p, v, bg, ba):
        arr = [np.ascontiguousarray(x, np.float64) for x in (q_xyzw, p, v, bg, ba)]
        _check(_lib.lvb_set_initial_state(self._h, seq, C.c_double(t), *[_p(a) for a in arr]))

    def get_state(self, seq):
        t = C.c_double()
        q = np.zeros(4); p = np.zeros(3); v = np.zeros(3); bg = np.zeros(3); ba = np.zeros(3)
        Pp = np.zeros((6, 6)); Pv = np.zeros((3, 3))
        _check(_lib.lvb_get_state(self._h, seq, C.byref(t), _p(q), _p(p), _p(v), _p(bg), _p(ba), _p(Pp), _p(Pv)))
        return dict(t=t.value, q=q, p=p, v=v, bg=bg, ba=ba, P_pose=Pp, P_vel=Pv)

    def get_calibration(self, seq):
        R = np.zeros((3, 3)); t = np.zeros(3); td = C.c_double(); Tg = np.zeros((3, 3)); As = np.zeros((3, 3)); Ma = np.zeros((3, 3))
        _check(_lib.lvb_get_calibration(self._h, seq, _p(R), _p(t), C.byref(td), _p(Tg), _p(As), _p(Ma)))
        return dict(R_imu_cam0=R, t_cam0_imu=t, td=td.value, Tg=Tg, As=As, Ma=Ma)

    def get_states(self):
        out = np.zeros((self.S, 17))
        _check(_lib.lvb_get_states(self._h, _p(out)))
        return out

    def get_covariance(self, seq, cap_dim=512):
        P = np.zeros((cap_dim, cap_dim))
        d = C.c_int()
        _check(_lib.lvb_get_covariance(self._h, seq, _p(P), cap_dim, C.byref(d)))
        n = d.value
        return P.reshape(-1)[:n * n].reshape(n, n).copy()

    def get_points(self, seq, which, cap=512):
        """which 0: stable (lost) map points, 1: active ones; returns {id: xyz} and clears the list (larvio.cpp:2719-2733)."""
        ids = np.zeros(cap, np.uint64); xyz = np.zeros((cap, 3)); n = C.c_int()
        _check(_lib.lvb_get_points(self._h, seq, int(which), _p(ids), _p(xyz), cap, C.byref(n)))
        return {int(ids[i]): xyz[i].copy() for i in range(n.value)}

    def get_window(self, seq, cap=64):
        qp = np.zeros((cap, 7)); n = C.c_int()
        _check(_lib.lvb_get_window(self._h, seq, _p(qp), cap, C.byref(n)))
        return qp[:n.value].copy()
