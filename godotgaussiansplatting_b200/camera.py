"""Host-side camera maths that the reference takes from the Godot engine.

* `perspective` restates Godot 4.3 `Projection::set_perspective` (engine source not vendored in the
  reference; stated from knowledge of Godot 4.x) -- what `Camera3D.get_camera_projection()` returns
  for the defaults fov 75, near 0.05, far 4000, keep_aspect = KEEP_HEIGHT (main.tscn:36-38).
* `pack_camera_push_constants` follows util/gaussian_splatting_rasterizer.gd:175-195 literally.
* `Camera3D` mirrors the handful of members the rasterizer touches (global_position,
  get_camera_transform, get_camera_projection); `reset()` follows util/camera.gd:151-153.
* `orbit_camera` generates the 1-degree-per-frame orbit of BASELINE.json config c3 (SURVEY 8d).
"""
from __future__ import annotations

import math

import numpy as np

F = np.float32


def perspective(fovy_degrees: float, aspect: float, z_near: float, z_far: float) -> np.ndarray:
    """Godot Projection columns x,y,z,w flattened (16 float32, column-major)."""
    radians = F(math.radians(F(fovy_degrees) / F(2.0)))
    delta_z = F(z_far) - F(z_near)
    sine = F(math.sin(radians))
    cotangent = F(F(math.cos(radians)) / sine)
    m = np.zeros((4, 4), dtype=np.float32)  # m[c][r]
    m[0][0] = cotangent / F(aspect)
    m[1][1] = cotangent
    m[2][2] = -(F(z_far) + F(z_near)) / delta_z
    m[2][3] = F(-1.0)
    m[3][2] = F(-2.0) * F(z_near) * F(z_far) / delta_z
    m[3][3] = F(0.0)
    return m.reshape(16)


def frustum(left: float, right: float, bottom: float, top: float, z_near: float, z_far: float) -> np.ndarray:
    """Godot `Projection.create_frustum` (Projection::set_frustum): an off-axis perspective with the near-plane window
    [left, right] x [bottom, top], as OpenXR hands each eye (XRInterface.get_projection_for_view).  16 float32, column-major.
    The off-centre terms sit in column z (m[2][0], m[2][1]): they shift a splat's image position by a constant per depth, and the EWA
    Jacobian of the projection reads only m[0][0] and m[1][1]."""
    l, r, b, t, n, f = (F(v) for v in (left, right, bottom, top, z_near, z_far))
    m = np.zeros((4, 4), dtype=np.float32)  # m[c][r]
    m[0][0] = F(2.0) * n / (r - l)
    m[1][1] = F(2.0) * n / (t - b)
    m[2][0] = (r + l) / (r - l)
    m[2][1] = (t + b) / (t - b)
    m[2][2] = -(f + n) / (f - n)
    m[2][3] = F(-1.0)
    m[3][2] = -(F(2.0) * f * n) / (f - n)
    return m.reshape(16)


def transform_to_projection(basis_cols: np.ndarray, origin: np.ndarray) -> np.ndarray:
    """Godot Projection(Transform3D): columns (x,0),(y,0),(z,0),(origin,1)."""
    m = np.zeros((4, 4), dtype=np.float32)
    m[0, :3], m[1, :3], m[2, :3] = basis_cols[0], basis_cols[1], basis_cols[2]
    m[3, :3] = origin
    m[3, 3] = 1.0
    return m.reshape(16)


def pack_camera_push_constants(view16: np.ndarray, proj16: np.ndarray) -> np.ndarray:
    """util/gaussian_splatting_rasterizer.gd:181-193 -> 32 float32 (view_matrix, projection_matrix)."""
    v = np.asarray(view16, dtype=np.float32).reshape(4, 4)
    p = np.asarray(proj16, dtype=np.float32).reshape(4, 4)
    x, y, z, w = v[0], v[1], v[2], v[3]

    def dot4(a, b):
        return ((a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]) + a[3] * b[3]

    out = np.array([
        -x[0], y[0], -z[0], 0.0,
        -x[1], y[1], -z[1], 0.0,
        x[2], -y[2], z[2], 0.0,
        -dot4(w, x), -dot4(w, -y), -dot4(w, z), 1.0,
        p[0][0], p[0][1], p[0][2], 0.0,
        p[1][0], p[1][1], p[1][2], 0.0,
        p[2][0], p[2][1], p[2][2], -1.0,
        p[3][0], p[3][1], p[3][2], 0.0], dtype=np.float32)
    return out


def _normalize(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v)


class Camera3D:
    """Minimal stand-in for Godot's Camera3D as used by the rasterizer (fov/near/far defaults of the engine)."""

    def __init__(self, fov: float = 75.0, near: float = 0.05, far: float = 4000.0):
        self.fov, self.near, self.far = float(fov), float(near), float(far)
        self.basis = np.eye(3, dtype=np.float32)  # rows of this array are the basis COLUMNS x, y, z
        self.global_position = np.zeros(3, dtype=np.float32)
        self.aspect = 16.0 / 9.0

    def reset(self) -> None:  # util/camera.gd:151-153: position = 0, rotation = UP * -PI
        self.global_position = np.zeros(3, dtype=np.float32)
        self.set_yaw(-math.pi)

    def set_yaw(self, yaw: float) -> None:
        c, s = F(math.cos(F(yaw))), F(math.sin(F(yaw)))
        # Basis rows [[c,0,s],[0,1,0],[-s,0,c]] -> columns x=(c,0,-s), y=(0,1,0), z=(s,0,c)
        self.basis = np.array([[c, 0, -s], [0, 1, 0], [s, 0, c]], dtype=np.float32)

    def look_at_from_position(self, position, target, up=(0.0, 1.0, 0.0)) -> None:
        """Node3D.look_at_from_position: -Z looks at target."""
        position = np.asarray(position, dtype=np.float64)
        vz = _normalize(position - np.asarray(target, dtype=np.float64))
        vx = _normalize(np.cross(np.asarray(up, dtype=np.float64), vz))
        vy = np.cross(vz, vx)
        self.basis = np.array([vx, vy, vz], dtype=np.float32)
        self.global_position = position.astype(np.float32)

    def get_camera_transform(self) -> np.ndarray:
        return transform_to_projection(self.basis, self.global_position)

    def get_camera_projection(self) -> np.ndarray:
        return perspective(self.fov, self.aspect, self.near, self.far)


def orbit_camera(frame: int, center=(0.0, 0.0, 2.5), radius: float = 2.5, pitch_deg: float = 10.0,
                 fov: float = 75.0, aspect: float = 16.0 / 9.0, step_deg: float = 1.0) -> Camera3D:
    """Camera for frame `frame` of the c3 orbit sweep: `step_deg` yaw steps about `center` at fixed radius
    and pitch, looking at the centroid.  Frame 0 sits at the c2 camera side (the world origin for the
    defaults), so frame 0 of the orbit sees the same view direction as the default camera."""
    yaw = math.radians(frame * step_deg)
    pitch = math.radians(pitch_deg)
    c = np.asarray(center, dtype=np.float64)
    # Godot world space shows the scene mirrored in x,y (rasterizer.gd:181-193); the centroid's x,y are
    # mirrored accordingly.  With the default centre (0,0,2.5) the mirror is a no-op.
    cw = np.array([-c[0], -c[1], c[2]])
    pos = cw + radius * np.array([math.sin(yaw) * math.cos(pitch), math.sin(pitch), -math.cos(yaw) * math.cos(pitch)])
    cam = Camera3D(fov=fov)
    cam.aspect = aspect
    cam.look_at_from_position(pos, cw)
    return cam


def stereo_pair(camera: Camera3D, ipd: float = 0.063) -> tuple[Camera3D, Camera3D]:
    """(left, right) eyes of `camera`: the same orientation and projection, positions offset by -ipd/2 and +ipd/2 along the
    camera's right axis (basis column x) -- what an XR runtime's per-view transforms are for a head pose."""
    eyes = []
    for sign in (-0.5, 0.5):
        e = Camera3D(fov=camera.fov, near=camera.near, far=camera.far)
        e.aspect = camera.aspect
        e.basis = camera.basis.copy()
        e.global_position = (camera.global_position.astype(np.float64) + sign * float(ipd) * camera.basis[0].astype(np.float64)).astype(np.float32)
        eyes.append(e)
    return eyes[0], eyes[1]


def default_camera(aspect: float = 16.0 / 9.0, fov: float = 75.0) -> Camera3D:
    cam = Camera3D(fov=fov)
    cam.aspect = aspect
    cam.reset()
    return cam


# ---------------------------------------------------------------------------------------------------------------------
# The application's own orbit (scope row f4): util/camera.gd FreeLookCamera -- set_focused_position (:144-149), the ORBIT
# branch of _input (:52-60) and the orbit branch of _update_movement (:127-137) once its 0.4 s ease-in is over (t = 1).
# ---------------------------------------------------------------------------------------------------------------------
def _rotated(v, axis, angle):
    """Vector3.rotated(axis, angle): Rodrigues' rotation about a unit axis."""
    v = np.asarray(v, dtype=np.float64)
    k = _normalize(axis)
    c, s = math.cos(angle), math.sin(angle)
    return v * c + np.cross(k, v) * s + k * np.dot(k, v) * (1.0 - c)


class FreeLookCamera(Camera3D):
    """util/camera.gd: the part that decides where the camera is while the user orbits a picked position.
    `target` is the $Target node the camera eases towards; in steady state (orbit_time >= 0.4, camera.gd:134) the camera's
    basis equals the target's and its position is the target position at the camera's current orbit radius."""

    def __init__(self, fov: float = 75.0, aspect: float = 16.0 / 9.0, mouse_sensitivity: float = 0.4):
        super().__init__(fov=fov)
        self.aspect = aspect
        self.mouse_sensitivity = float(mouse_sensitivity)          # camera.gd:5
        self.target = Camera3D(fov=fov)                             # $Target (a Node3D: only basis + position are used)
        self.reset()

    def reset(self) -> None:                                        # camera.gd:151-159
        super().reset()
        self.orbit_position = np.array([0.0, 0.0, 2.0])             # -Vector3.FORWARD * 2.0
        self.target.basis = np.eye(3, dtype=np.float32)
        self.target.global_position = np.zeros(3, dtype=np.float32)

    def set_focused_position(self, target_position) -> None:        # camera.gd:144-149 (main.gd:89-91 calls it with the picked splat)
        self.orbit_position = np.asarray(target_position, dtype=np.float64)
        # $Target is top_level (main.tscn:53-54): its position is global -- two units from the focus along the camera's view axis
        self.target.global_position = (self.orbit_position + self.basis[2].astype(np.float64) * 2.0).astype(np.float32)
        # :140-141 the camera eases to target.position; then, holding the orbit button, OrbitSwapTimer (:38-43) makes the target look at
        # the focus from there and the camera eases into the target's orientation (:127-137).  Steady state of both:
        self.global_position = self.target.global_position.copy()
        self.target.look_at_from_position(self.global_position.astype(np.float64), self.orbit_position)
        self.basis = self.target.basis.copy()

    def _target_pitch_deg(self) -> float:
        """target.rotation_degrees.x: Euler YXZ of a roll-free look-at basis = asin(-basis.z.y)."""
        return math.degrees(math.asin(max(-1.0, min(1.0, -float(self.target.basis[2][1])))))

    def orbit_mouse_motion(self, relative_x: float, relative_y: float) -> None:
        """InputEventMouseMotion in RotationMode.ORBIT (camera.gd:52-60), then one _process tick in steady state (:127-137, t = 1)."""
        off_x, off_y = -relative_x * self.mouse_sensitivity, -relative_y * self.mouse_sensitivity      # :49
        pitch = self._target_pitch_deg() - off_y                                                       # :53
        tp = self.target.global_position.astype(np.float64)
        rotated = tp - self.orbit_position                                                             # :54
        tb = self.target.basis.astype(np.float64)
        if -80.0 <= pitch <= 70.0:                                                                     # :55-56
            rotated = _rotated(rotated, tb[0], math.radians(-off_y))
        rotated = _rotated(rotated, tb[1], math.radians(-off_x) * math.cos(math.radians(pitch)))      # :57
        rotated = rotated + self.orbit_position                                                        # :58
        self.target.look_at_from_position(rotated, self.orbit_position)                                # :59
        # _update_movement, orbit branch with t = 1: the camera takes the target's orientation and the target's direction
        # from the orbit position at its own current radius (:129-137)
        radius = float(np.linalg.norm(self.orbit_position - self.global_position.astype(np.float64)))
        d = _normalize(self.target.global_position.astype(np.float64) - self.orbit_position)
        self.basis = self.target.basis.copy()
        self.global_position = (self.orbit_position + d * radius).astype(np.float32)
        # :140-141 smooth distance transition towards target.position: in steady state the camera has arrived
        self.global_position = self.target.global_position.copy()


def reference_orbit_sweep(n_frames: int, focus=(0.0, 0.0, 2.5), yaw_step_deg: float = 1.0, start_pitch_deg: float = -10.0, zoom_clicks: int = 2,
                          fov: float = 75.0, aspect: float = 16.0 / 9.0):
    """The c3 sweep driven the way the application drives it: focus the camera on `focus` (a picked splat position, main.gd:86-91),
    then one mouse-motion event per frame whose horizontal movement turns the view by `yaw_step_deg` about the focus
    (camera.gd:57: the yaw applied is offset.x * cos(pitch), so the event carries yaw_step / (sensitivity * cos(pitch)))."""
    cam = FreeLookCamera(fov=fov, aspect=aspect)
    cam.set_focused_position(focus)
    for _ in range(zoom_clicks):   # MOUSE_BUTTON_WHEEL_DOWN (:76-78): the target backs off the focus by 0.25 per click, the camera follows (:140-141)
        tp = cam.target.global_position.astype(np.float64)
        cam.target.global_position = (tp - _normalize(cam.orbit_position - tp) * 0.25).astype(np.float32)
        cam.global_position = cam.target.global_position.copy()
    if start_pitch_deg:
        cam.orbit_mouse_motion(0.0, -start_pitch_deg / cam.mouse_sensitivity * -1.0)   # one vertical drag to the starting pitch
    out = []
    for _ in range(n_frames):
        out.append((cam.get_camera_transform(), cam.get_camera_projection(), cam.global_position.copy()))
        pitch = cam._target_pitch_deg()
        cam.orbit_mouse_motion(-yaw_step_deg / (cam.mouse_sensitivity * math.cos(math.radians(pitch))), 0.0)
    return out
