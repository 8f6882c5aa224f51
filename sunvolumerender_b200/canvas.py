"""Python mirror of include/svr_canvas.h: the reference's Canvas (gui/canvas.{h,cpp}) without its window.
`View` is the camera manipulation as host arithmetic (no GPU needed); `Canvas` owns the frame buffers, forwards
setters to the setup_* entry points, restarts the progressive render and paints frames."""
import ctypes as C

import numpy as np

from . import _lib as L


def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


class View:
    def __init__(self, width, height):
        self.lib = L.load()
        self.width, self.height = int(width), int(height)
        self.v = L.View()
        self.lib.svr_view_init(C.byref(self.v))

    def reset(self, volume_size):
        self.lib.svr_view_reset(C.byref(self.v), C.byref(_f3(volume_size)))

    def zoom_to_extent(self, volume_size):
        self.lib.svr_view_zoom_to_extent(C.byref(self.v), C.byref(_f3(volume_size)))

    def rotate(self, degrees, axis):
        self.lib.svr_view_rotate(C.byref(self.v), degrees, *[float(a) for a in axis])

    def mouse_press(self, px, py, buttons):
        return self.lib.svr_view_mouse_press(C.byref(self.v), self.width, self.height, px, py, buttons)

    def mouse_move(self, px, py, buttons, volume_size):
        return self.lib.svr_view_mouse_move(C.byref(self.v), self.width, self.height, px, py, buttons, C.byref(_f3(volume_size)))

    def wheel(self, delta, volume_size):
        return self.lib.svr_view_wheel(C.byref(self.v), int(delta), C.byref(_f3(volume_size)))

    def key(self, key):
        return self.lib.svr_view_key(C.byref(self.v), key)

    def camera(self):
        cam = L.Camera()
        self.lib.svr_view_camera(C.byref(self.v), self.width, self.height, C.byref(cam))
        return cam

    def matrix(self):
        """glm::mat4 as m[c][r]."""
        return np.array(list(self.v.viewMat), np.float32).reshape(4, 4)


class Canvas:
    """Needs a CUDA device (the entry points it drives have no CPU path)."""

    def __init__(self, width, height):
        self.lib = L.load()
        self.width, self.height = int(width), int(height)
        self.c = self.lib.svr_canvas_create(self.width, self.height)
        if not self.c:
            raise L.SvrError("svr_canvas_create failed: " + self.lib.svr_last_error().decode())

    def close(self):
        if self.c:
            self.lib.svr_canvas_destroy(self.c)
            self.c = None

    def _ck(self, rc, what):
        L.check(rc, what)

    # ---- scene
    def load_volume(self, path):
        self._ck(self.lib.svr_canvas_load_volume(self.c, str(path).encode()), "svr_canvas_load_volume")

    def set_volume(self, volume, volume_size, element_radius):
        self._ck(self.lib.svr_canvas_set_volume(self.c, C.byref(volume), C.byref(_f3(volume_size)), element_radius), "svr_canvas_set_volume")

    def set_transfer_function(self, tf):
        self._ck(self.lib.svr_canvas_set_transfer_function(self.c, C.byref(tf)), "svr_canvas_set_transfer_function")

    def set_area_lights(self, lights):
        arr = (L.AreaLight * max(1, len(lights)))(*lights)
        self._ck(self.lib.svr_canvas_set_area_lights(self.c, arr, len(lights)), "svr_canvas_set_area_lights")

    def set(self, **kw):
        """density_scale, gradient_factor, scatter_times, render_mode, env_background=(r,g,b), env_map=path,
        env_offset=(u,v), env_intensity, fov, apeture, focal_length, exposure, x_clip / y_clip / z_clip=(lo,hi)"""
        lib, c = self.lib, self.c
        for k, v in kw.items():
            if k in ("x_clip", "y_clip", "z_clip"):
                rc = lib.svr_canvas_set_clip_plane(c, "xyz".index(k[0]), v[0], v[1])
            elif k == "env_background":
                rc = lib.svr_canvas_set_env_background(c, *[float(x) for x in v])
            elif k == "env_offset":
                rc = lib.svr_canvas_set_env_offset(c, float(v[0]), float(v[1]))
            elif k == "env_map":
                rc = lib.svr_canvas_set_env_map(c, str(v).encode())
            else:
                rc = getattr(lib, "svr_canvas_set_" + k)(c, v)
            self._ck(rc, "svr_canvas_set_" + k)

    def set_projection(self, mode="max", window=(0.5, 1.0)):
        """Projection mode's settings (svr_canvas_set_projection): mode "max", "min" or "mean", window (center, width);
        select the mode with set(render_mode=L.RENDER_MODE_PROJECTION)."""
        self._ck(self.lib.svr_canvas_set_projection(self.c, L.PROJECT_MODES[mode], float(window[0]), float(window[1])), "svr_canvas_set_projection")

    def set_immediate_repaint(self, on):
        self.lib.svr_canvas_set_immediate_repaint(self.c, 1 if on else 0)

    # ---- events
    def mouse_press(self, px, py, buttons):
        self._ck(self.lib.svr_canvas_mouse_press(self.c, px, py, buttons), "svr_canvas_mouse_press")

    def mouse_move(self, px, py, buttons):
        self._ck(self.lib.svr_canvas_mouse_move(self.c, px, py, buttons), "svr_canvas_mouse_move")

    def wheel(self, delta):
        self._ck(self.lib.svr_canvas_wheel(self.c, int(delta)), "svr_canvas_wheel")

    def key(self, key):
        self._ck(self.lib.svr_canvas_key(self.c, key), "svr_canvas_key")

    # ---- frames
    def paint(self, n=1):
        for _ in range(n):
            self._ck(self.lib.svr_canvas_paint(self.c), "svr_canvas_paint")

    def image(self):
        out = np.zeros((self.height, self.width, 4), np.uint8)
        self._ck(self.lib.svr_canvas_read_image(self.c, C.c_void_p(out.ctypes.data)), "svr_canvas_read_image")
        return out

    @property
    def frame_no(self):
        return int(self.lib.svr_canvas_frame_no(self.c))

    @property
    def paint_count(self):
        return int(self.lib.svr_canvas_paint_count(self.c))

    def camera(self):
        cam = L.Camera()
        self.lib.svr_canvas_get_camera(self.c, C.byref(cam))
        return cam

    def view(self):
        v = L.View()
        self.lib.svr_canvas_get_view(self.c, C.byref(v))
        return v

    def volume(self):
        v = L.Volume()
        self.lib.svr_canvas_get_volume(self.c, C.byref(v))
        return v

    def env_light(self):
        e = L.EnvLight()
        self.lib.svr_canvas_get_env_light(self.c, C.byref(e))
        return e

    def hdr_ptr(self):
        return self.lib.svr_canvas_hdr(self.c)

    def image_ptr(self):
        return self.lib.svr_canvas_image(self.c)
