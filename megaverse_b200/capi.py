"""ctypes binding of the C ABI (include/megaverse_b200.h).  This is the reference-side stub INTEGRATION.md describes: what a
maintainer would bind from Python if they did not want the pybind11 module.  It loads the in-tree libmegaverse_b200.so and
fails loudly when the library or a CUDA device is missing -- there is no CPU fallback in the product."""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MV_B200_LIB") or os.path.join(_PKG, "libmegaverse_b200.so")  # the override is for kernel-variant experiments (tools/)
_lib = None

MV_OK, MV_ERR_ARG, MV_ERR_CUDA, MV_ERR_CAPACITY, MV_ERR_STATE = 0, -1, -2, -3, -4


class MegaverseError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("megaverse_b200 error %d: %s" % (code, msg))
        self.code = code


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: run `python -m megaverse_b200._build` (needs nvcc)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, ci, cf = C.c_void_p, C.c_int, C.c_float
        L.mv_create.argtypes = [C.c_char_p, ci, ci, ci, ci, ci, ci, C.POINTER(C.c_char_p), C.POINTER(cf), ci, C.POINTER(vp)]
        L.mv_last_error.argtypes = [vp]
        L.mv_last_error.restype = C.c_char_p
        for name in ("mv_reset", "mv_step", "mv_step_begin", "mv_step_end", "mv_close", "mv_sync", "mv_fetch_obs"):
            getattr(L, name).argtypes = [vp]
        L.mv_seed.argtypes = [vp, ci]
        L.mv_seed_env.argtypes = [vp, ci, ci]
        L.mv_set_actions.argtypes = [vp, vp]
        L.mv_encode_action.argtypes = [vp]
        L.mv_step_device.argtypes = [vp, vp]
        for name in ("mv_obs_host", "mv_depth_host", "mv_rewards", "mv_dones", "mv_true_objectives", "mv_actions_device", "mv_obs_device",
                     "mv_depth_device", "mv_rewards_device", "mv_dones_device", "mv_stream"):
            getattr(L, name).argtypes = [vp, C.POINTER(vp)]
        L.mv_get_reward_shaping.argtypes = [vp, ci, ci, C.POINTER(C.c_char_p), C.POINTER(cf), ci, C.POINTER(ci)]
        L.mv_set_reward_shaping.argtypes = [vp, ci, ci, C.POINTER(C.c_char_p), C.POINTER(cf), ci]
        L.mv_set_option.argtypes = [vp, C.c_char_p, ci]
        L.mv_faults.argtypes = [vp, C.POINTER(C.c_int32)]
        L.mv_kernel_launches.argtypes = [vp, C.POINTER(C.c_int64)]
        L.mv_last_kernel_ms.argtypes = [vp, C.POINTER(cf)]
        for name in ("mv_debug_get_level", "mv_debug_get_state", "mv_debug_get_voxels", "mv_debug_get_instances"):
            getattr(L, name).argtypes = [vp, ci, vp, ci]
        L.mv_debug_get_view.argtypes = [vp, ci, ci, vp]
        L.mv_debug_render_instances.argtypes = [vp, vp, ci, ci, ci, vp, vp]
        L.mv_debug_bzset.argtypes = [vp, ci, vp, ci]
        L.mv_debug_generate_level.argtypes = [C.c_char_p, ci, ci, ci, C.POINTER(C.c_char_p), C.POINTER(cf), ci, vp, ci]
        _lib = L
    return _lib


EXPORTS = [
    "mv_create", "mv_last_error", "mv_seed", "mv_seed_env", "mv_reset", "mv_set_actions", "mv_encode_action", "mv_step", "mv_step_begin", "mv_step_end", "mv_obs_host", "mv_depth_host",
    "mv_rewards", "mv_dones", "mv_true_objectives", "mv_get_reward_shaping", "mv_set_reward_shaping", "mv_set_option", "mv_step_device", "mv_set_obs_buffer",
    "mv_sync", "mv_fetch_obs", "mv_draw_hires", "mv_actions_device", "mv_obs_device", "mv_depth_device", "mv_rewards_device", "mv_dones_device", "mv_stream", "mv_faults", "mv_fault_word", "mv_kernel_launches",
    "mv_last_kernel_ms", "mv_close", "mv_debug_get_level", "mv_debug_get_state", "mv_debug_get_voxels", "mv_debug_get_instances", "mv_debug_get_view",
    "mv_debug_render_instances", "mv_debug_step_profile", "mv_debug_raster_config", "mv_debug_static_cap", "mv_debug_raster_stats", "mv_debug_color_tables", "mv_debug_defaults", "mv_debug_count_unfit_levels", "mv_levels_skipped", "mv_debug_bzset", "mv_debug_generate_level",
]


class Engine:
    """Thin object wrapper: one method per C entry point, numpy views over engine-owned host memory."""

    def __init__(self, scenario, num_envs, num_agents, w=128, h=72, num_threads=1, device=0, params=None, depth=False):
        L = lib()
        params = params or {}
        keys = (C.c_char_p * max(1, len(params)))(*[k.encode() for k in params])
        vals = (C.c_float * max(1, len(params)))(*[float(v) for v in params.values()])
        self._h = C.c_void_p()
        rc = L.mv_create(scenario.encode(), w, h, num_envs, num_agents, num_threads, device, keys, vals, len(params), C.byref(self._h))
        if rc != MV_OK:
            raise MegaverseError(rc, (L.mv_last_error(None) or b"").decode())
        self.E, self.A, self.N, self.w, self.h = num_envs, num_agents, num_envs * num_agents, w, h
        if depth:
            self._ck(L.mv_set_option(self._h, b"depth", 1))

    def _ck(self, rc):
        if rc != MV_OK:
            raise MegaverseError(rc, (lib().mv_last_error(self._h) or b"").decode())

    def close(self):
        if self._h:
            lib().mv_close(self._h)
            self._h = C.c_void_p()

    def set_option(self, key, value):
        self._ck(lib().mv_set_option(self._h, key.encode(), int(value)))

    def seed(self, s):
        self._ck(lib().mv_seed(self._h, int(s)))

    def seed_env(self, e, s):
        self._ck(lib().mv_seed_env(self._h, int(e), int(s)))

    def reset(self):
        self._ck(lib().mv_reset(self._h))

    def step(self, masks):
        m = np.ascontiguousarray(masks, dtype=np.int32)
        assert m.size == self.N
        self._ck(lib().mv_set_actions(self._h, m.ctypes.data))
        self._ck(lib().mv_step(self._h))

    def step_begin(self, masks):
        """first half of step(): upload the masks, enqueue kernels and device->host copies, return at once"""
        m = np.ascontiguousarray(masks, dtype=np.int32)
        assert m.size == self.N
        self._ck(lib().mv_set_actions(self._h, m.ctypes.data))
        self._ck(lib().mv_step_begin(self._h))

    def step_end(self):
        """second half: wait; obs() / rewards() / dones() are then valid as after step()"""
        self._ck(lib().mv_step_end(self._h))

    def step_device(self, d_masks_ptr=None):
        self._ck(lib().mv_step_device(self._h, C.c_void_p(d_masks_ptr) if d_masks_ptr else None))

    def set_obs_buffer(self, d_obs_ptr=None, d_depth_ptr=None):
        """rasterise into caller-owned device memory (a slice of a larger tensor) instead of the engine's own obs buffer"""
        lib().mv_set_obs_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        self._ck(lib().mv_set_obs_buffer(self._h, C.c_void_p(d_obs_ptr) if d_obs_ptr else None, C.c_void_p(d_depth_ptr) if d_depth_ptr else None))

    def sync(self):
        self._ck(lib().mv_sync(self._h))

    def draw_hires(self, w, h):
        """uint8[N,h,w,4] view of the engine's hi-res frame (valid until the next draw_hires)"""
        p = C.c_void_p()
        lib().mv_draw_hires.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        self._ck(lib().mv_draw_hires(self._h, int(w), int(h), C.byref(p)))
        n = self.N * h * w * 4
        return np.frombuffer((C.c_char * n).from_address(p.value), dtype=np.uint8).reshape(self.N, h, w, 4)

    def device_array(self, what="obs"):
        """zero-copy handle on an engine-owned device tensor for any consumer of the CUDA array interface
        (`torch.as_tensor(eng.device_array("obs"), device="cuda")`, CuPy, Numba): "obs" uint8[N,h,w,4], "depth" float32[N,h,w],
        "rewards" float32[N], "dones" uint8[E].  Valid in the engine stream's order (mv_stream) until mv_close."""
        shapes = {"obs": ((self.N, self.h, self.w, 4), "|u1"), "depth": ((self.N, self.h, self.w), "<f4"), "rewards": ((self.N,), "<f4"), "dones": ((self.E,), "|u1")}
        shape, typestr = shapes[what]
        ptr, stream = self.device_ptr(what), self.stream()

        class _DeviceArray:
            __cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 3, "strides": None, "stream": stream or 1}

        return _DeviceArray()

    def fetch_obs(self):
        self._ck(lib().mv_fetch_obs(self._h))

    def _host(self, fn, shape, dtype):
        p = C.c_void_p()
        self._ck(getattr(lib(), fn)(self._h, C.byref(p)))
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        return np.frombuffer((C.c_char * n).from_address(p.value), dtype=dtype).reshape(shape)

    def obs(self):
        """uint8[N,h,w,4]: a VIEW of engine memory, valid until the next step (megaverse.cpp:139-143)"""
        return self._host("mv_obs_host", (self.N, self.h, self.w, 4), np.uint8)

    def depth(self):
        return self._host("mv_depth_host", (self.N, self.h, self.w), np.float32)

    def rewards(self):
        return self._host("mv_rewards", (self.N,), np.float32)

    def dones(self):
        return self._host("mv_dones", (self.E,), np.uint8)

    def true_objectives(self):
        return self._host("mv_true_objectives", (self.N,), np.float32)

    def device_ptr(self, what):
        p = C.c_void_p()
        self._ck(getattr(lib(), "mv_%s_device" % what)(self._h, C.byref(p)))
        return p.value

    def stream(self):
        p = C.c_void_p()
        self._ck(lib().mv_stream(self._h, C.byref(p)))
        return p.value

    def get_reward_shaping(self, env, agent):
        keys = (C.c_char_p * 32)()
        vals = (C.c_float * 32)()
        n = C.c_int()
        self._ck(lib().mv_get_reward_shaping(self._h, env, agent, keys, vals, 32, C.byref(n)))
        return {keys[i].decode(): float(vals[i]) for i in range(n.value)}

    def set_reward_shaping(self, env, agent, rs):
        keys = (C.c_char_p * max(1, len(rs)))(*[k.encode() for k in rs])
        vals = (C.c_float * max(1, len(rs)))(*[float(v) for v in rs.values()])
        self._ck(lib().mv_set_reward_shaping(self._h, env, agent, keys, vals, len(rs)))

    def faults(self):
        f = C.c_int32()
        self._ck(lib().mv_faults(self._h, C.byref(f)))
        return f.value

    def fault_word(self):
        """the latched fault bits without a device round trip (mv_fault_word)"""
        f = C.c_int32()
        lib().mv_fault_word.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
        self._ck(lib().mv_fault_word(self._h, C.byref(f)))
        return f.value

    def kernel_launches(self):
        n = C.c_int64()
        self._ck(lib().mv_kernel_launches(self._h, C.byref(n)))
        return n.value

    def step_profile(self, enable=True, read=True):
        out = np.zeros((self.E, 16), dtype=np.uint32)
        lib().mv_debug_step_profile.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        self._ck(lib().mv_debug_step_profile(self._h, out.ctypes.data if read else None, 1 if enable else 0))
        return out

    def static_cap(self):
        lib().mv_debug_static_cap.argtypes = [C.c_void_p]
        return int(lib().mv_debug_static_cap(self._h))

    def raster_config(self):
        out = (C.c_int32 * 4)()
        lib().mv_debug_raster_config.argtypes = [C.c_void_p, C.c_void_p]
        self._ck(lib().mv_debug_raster_config(self._h, out))
        return {"grid": out[0], "ctas_per_sm": out[1], "smem": out[2], "bands": out[3]}

    def raster_stats(self, enable=True, read=True):
        out = (C.c_ulonglong * 16)()
        lib().mv_debug_raster_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        self._ck(lib().mv_debug_raster_stats(self._h, out if read else None, 1 if enable else 0))
        names = ["work_items", "instances", "visible_instances", "items", "clipped_items", "triangles", "batches", "sub_passes", "cyc_head", "cyc_tma_wait", "cyc_instance", "cyc_item", "cyc_tile", "cyc_total",
                 "pairs_evaluated", "pairs_in_boxes"]  # (tile, triangle) pairs: kept by the binning / in the triangles' pixel boxes
        return {n: int(out[i]) for i, n in enumerate(names)}

    def last_kernel_ms(self):
        out = (C.c_float * 2)()
        self._ck(lib().mv_last_kernel_ms(self._h, out))
        return float(out[0]), float(out[1])

    # ---- introspection (tests)
    def _dump(self, fn, env, dtype, cap=1 << 16):
        out = np.zeros(cap, dtype=dtype)
        n = getattr(lib(), fn)(self._h, env, out.ctypes.data, cap)
        if n < -8:
            return self._dump(fn, env, dtype, -n)
        if n < 0:
            self._ck(n)
        return out[:n].copy()

    def level(self, env):
        return self._dump("mv_debug_get_level", env, np.int32)

    def state(self, env):
        return self._dump("mv_debug_get_state", env, np.float32)

    def voxels(self, env):
        return self._dump("mv_debug_get_voxels", env, np.int32).reshape(-1, 4)

    def instances(self, env):
        return self._dump("mv_debug_get_instances", env, np.float32).reshape(-1, 18)

    def view(self, env, agent):
        out = np.zeros(16, dtype=np.float32)
        self._ck(lib().mv_debug_get_view(self._h, env, agent, out.ctypes.data))
        return out


def render_instances(view16, inst18, w, h, want_depth=False):
    view16 = np.ascontiguousarray(view16, dtype=np.float32)
    inst18 = np.ascontiguousarray(inst18, dtype=np.float32).reshape(-1, 18)
    rgba = np.zeros((h, w, 4), dtype=np.uint8)
    depth = np.zeros((h, w), dtype=np.float32)
    rc = lib().mv_debug_render_instances(view16.ctypes.data, inst18.ctypes.data, inst18.shape[0], w, h, rgba.ctypes.data, depth.ctypes.data if want_depth else None)
    if rc != MV_OK:
        raise MegaverseError(rc, "mv_debug_render_instances failed")
    return (rgba, depth) if want_depth else rgba


def generate_level(scenario, num_agents, env_seed, episode, params=None):
    """host-only level generation (no CUDA): int32 dump of episode `episode` of the env stream seeded with env_seed"""
    params = params or {}
    keys = (C.c_char_p * max(1, len(params)))(*[k.encode() for k in params])
    vals = (C.c_float * max(1, len(params)))(*[float(v) for v in params.values()])
    out = np.zeros(1 << 14, dtype=np.int32)
    n = lib().mv_debug_generate_level(scenario.encode(), num_agents, env_seed, episode, keys, vals, len(params), out.ctypes.data, out.size)
    if n < 0:
        raise MegaverseError(n, "mv_debug_generate_level failed")
    return out[:n].copy()


def bzset_order(ops):
    ops = np.ascontiguousarray(ops, dtype=np.int32).reshape(-1, 4)
    out = np.zeros(3 * 256, dtype=np.int32)
    n = lib().mv_debug_bzset(ops.ctypes.data, ops.shape[0], out.ctypes.data, out.size)
    return out[: n * 3].reshape(n, 3).copy()


def encode_action(heads6):
    a = np.ascontiguousarray(heads6, dtype=np.int32)
    return int(lib().mv_encode_action(a.ctypes.data))
