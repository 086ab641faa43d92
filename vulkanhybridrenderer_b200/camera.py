"""Camera / per-frame constants of the headless harness.

Reproduces the reference's recipe:
  * projection: VkUtils::InfiniteReverseDepthProjection (/root/reference/src/rendering_backend/vulkan_utils.h:494-503)
  * camera transform/view: scene_loader.cpp:43-71 (transform = T * yawPitchRoll, view = inverse(transform))
  * PerFrameData fill: renderer.cpp:187-204
  * directional light: scene_loader.cpp:74-99

Math is done on ordinary row-major 4x4 numpy matrices (M[r, c]); `to_glm` transposes into the column-major
storage of glsl_common.h when the struct is filled.
"""
import numpy as np

from . import types as T


def to_glm(m):
    return np.ascontiguousarray(np.asarray(m, dtype=np.float32).T)


def infinite_reverse_depth_projection(yfov, aspect, znear):
    s = np.float32(1.0) / np.tan(np.float32(yfov) * np.float32(0.5))
    m = np.zeros((4, 4), np.float32)
    m[0, 0] = s / np.float32(aspect)
    m[1, 1] = s
    m[3, 2] = -1.0          # column 2 = (0,0,0,-1)
    m[2, 3] = znear         # column 3 = (0,0,znear,0)
    return m


def yaw_pitch_roll(yaw, pitch, roll=0.0):
    """glm::yawPitchRoll (Y * X * Z)."""
    cy, sy = np.cos(yaw), np.sin(yaw)
    cp, sp = np.cos(pitch), np.sin(pitch)
    cr, sr = np.cos(roll), np.sin(roll)
    ry = np.array([[cy, 0, sy, 0], [0, 1, 0, 0], [-sy, 0, cy, 0], [0, 0, 0, 1]], np.float64)
    rx = np.array([[1, 0, 0, 0], [0, cp, -sp, 0], [0, sp, cp, 0], [0, 0, 0, 1]], np.float64)
    rz = np.array([[cr, -sr, 0, 0], [sr, cr, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1]], np.float64)
    return ry @ rx @ rz


def camera_transform(position, yaw, pitch, roll=0.0):
    t = np.eye(4)
    t[:3, 3] = position
    return (t @ yaw_pitch_roll(yaw, pitch, roll)).astype(np.float32)


class Camera:
    """Camera with the fields of the reference's `Camera` (transform, view, perspective)."""

    def __init__(self, position, yaw, pitch, yfov, aspect, znear=0.1):
        self.yfov, self.aspect, self.znear = yfov, aspect, znear
        self.perspective = infinite_reverse_depth_projection(yfov, aspect, znear)
        self.set_pose(position, yaw, pitch)

    def set_pose(self, position, yaw, pitch):
        self.position = np.asarray(position, np.float64)
        self.yaw, self.pitch = yaw, pitch
        self.transform = camera_transform(self.position, yaw, pitch)
        self.view = np.linalg.inv(self.transform.astype(np.float64)).astype(np.float32)


def directional_light(direction, color=(1.0, 1.0, 1.0), intensity=30.0):
    dl = np.zeros((), T.DirectionalLight)
    d = np.asarray(direction, np.float64)
    d = d / np.linalg.norm(d)
    dl["projview"] = np.eye(4, dtype=np.float32)      # only read by the rasterised shadow map (out of scope)
    dl["direction"] = (d[0], d[1], d[2], 0.0)
    dl["color"] = (color[0], color[1], color[2], 1.0)
    dl["intensity"] = (intensity,) * 4
    return dl


def _ortho_reverse_z(l, r, b, t, zn, zf):
    """glm::orthoRH_ZO(l, r, b, t, zn, zf) (GLM_FORCE_DEPTH_ZERO_TO_ONE): with zn > zf, depth 0 at distance zn, 1 at zf."""
    p = np.eye(4)
    p[0, 0], p[1, 1], p[2, 2] = 2.0 / (r - l), 2.0 / (t - b), -1.0 / (zf - zn)
    p[0, 3], p[1, 3], p[2, 3] = -(r + l) / (r - l), -(t + b) / (t - b), -zn / (zf - zn)
    return p


def _look_at(eye, center, up):
    """glm::lookAtRH"""
    f = np.asarray(center, np.float64) - eye
    f = f / np.linalg.norm(f)
    s = np.cross(f, up)
    s = s / np.linalg.norm(s)
    u = np.cross(s, f)
    v = np.eye(4)
    v[0, :3], v[1, :3], v[2, :3] = s, u, -f
    v[0, 3], v[1, 3], v[2, 3] = -s @ eye, -u @ eye, f @ eye
    return v


def light_projview(direction):
    """directional_light.projview as the reference's scene loader builds it (scene_loader.cpp:74-100, host/scene_loader.cpp
    setup_directional_light): glm::ortho(-8, 8, -8, 8, 12, 0.1) * glm::lookAt(-12 d, 0, +y), column-major float32. The window is
    fixed: depth 0 lies on the plane through the origin, so geometry farther from the light than the origin is clipped."""
    d = np.asarray(direction, np.float64)[:3]
    d = d / np.linalg.norm(d)
    pv = _ortho_reverse_z(-8.0, 8.0, -8.0, 8.0, 12.0, 0.1) @ _look_at(-12.0 * d, np.zeros(3), np.array([0.0, 1.0, 0.0]))
    return to_glm(pv)


def fit_light_projview(direction, scene_min, scene_max, margin=0.01):
    """Test and timing harness only (the reference has no such matrix): the same ortho * lookAt form, with a window and near / far
    planes that enclose the box [scene_min, scene_max] seen along `direction` (plus `margin` of its diagonal), so that nothing is
    clipped. Depth 1 is the nearest point of the box, 0 the farthest."""
    d = np.asarray(direction, np.float64)[:3]
    d = d / np.linalg.norm(d)
    lo, hi = np.asarray(scene_min, np.float64), np.asarray(scene_max, np.float64)
    c, r = 0.5 * (lo + hi), 0.5 * np.linalg.norm(hi - lo)
    up = np.array([0.0, 1.0, 0.0]) if abs(d[1]) < 0.999 else np.array([0.0, 0.0, 1.0])
    view = _look_at(c - d * (r + 1.0), c, up)
    corners = np.array([[x, y, z, 1.0] for x in (lo[0], hi[0]) for y in (lo[1], hi[1]) for z in (lo[2], hi[2])]) @ view.T
    pad = margin * 2.0 * r + 1e-6
    (x0, y0), (x1, y1) = corners[:, :2].min(0) - pad, corners[:, :2].max(0) + pad
    dist = -corners[:, 2]
    pv = _ortho_reverse_z(x0, x1, y0, y1, dist.max() + pad, dist.min() - pad) @ view
    return to_glm(pv)


class FrameSequencer:
    """renderer.cpp:187-204: keeps last frame's view/proj and the post-incremented frame index.

    The reference starts at frame_index 0 with zero previous matrices (SURVEY Q5: NaN motion vectors, one seed for
    every pixel). The harness starts at `first_frame_index` (default 1) with prev = current so frame 0 of a test is
    well defined; both are documented deviations of the harness, not of the kernels.
    """

    def __init__(self, width, height, light, first_frame_index=1):
        self.width, self.height = width, height
        self.light = light
        self.frame_index = first_frame_index
        self.prev_view = None
        self.prev_proj = None

    def next(self, camera):
        pfd = np.zeros((), T.PerFrameData)
        view = camera.view
        proj = camera.perspective
        pfd["camera_view"] = to_glm(view)
        pfd["camera_proj"] = to_glm(proj)
        pfd["camera_view_inverse"] = to_glm(camera.transform)
        pfd["camera_proj_inverse"] = to_glm(np.linalg.inv(proj.astype(np.float64)))
        pfd["camera_viewproj_inverse"] = to_glm(np.linalg.inv(proj.astype(np.float64) @ view.astype(np.float64)))
        pv = view if self.prev_view is None else self.prev_view
        pp = proj if self.prev_proj is None else self.prev_proj
        pfd["camera_view_prev_frame"] = to_glm(pv)
        pfd["camera_proj_prev_frame"] = to_glm(pp)
        pfd["directional_light"] = self.light
        pfd["display_size"] = (self.width, self.height)
        pfd["display_size_inverse"] = (np.float32(1.0) / np.float32(self.width), np.float32(1.0) / np.float32(self.height))
        pfd["frame_index"] = self.frame_index
        pfd["blue_noise_texture_index"] = -1
        self.frame_index += 1
        self.prev_view, self.prev_proj = view.copy(), proj.copy()
        return pfd
