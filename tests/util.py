"""Shared seeded test problems (inputs only; expected values always come from the oracle or golden files)."""
import hashlib
import json
import os

import numpy as np

from direct_visual_lidar_calibration_b200 import synthetic as S

REFERENCE_OUTPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.json")

# model -> (intrinsics, distortion, (W, H))
CAMERAS = {
    "plumb_bob": ([400.0, 410.0, 320.0, 240.0], [-0.04, 0.08, 1e-4, -3e-4, -0.04], (640, 480)),
    "fisheye": ([300.0, 300.0, 320.0, 240.0], [0.01, -0.02, 0.003, -0.001], (640, 480)),
    "atan": ([400.0, 400.0, 320.0, 240.0], [0.9], (640, 480)),
    "omnidir": ([300.0, 300.0, 320.0, 240.0, 1.1], [-0.1, 0.02, 1e-3, -2e-3], (640, 480)),
    "equirectangular": ([640.0, 320.0], [], (640, 320)),
    "rational_polynomial": ([400.0, 410.0, 320.0, 240.0], [-0.04, 0.08, 1e-4, -3e-4, -0.04, 0.01, 0.02, -0.005], (640, 480)),
}
MODELS = list(CAMERAS.keys())


def random_problem(model, n=20000, seed=0, size=None, f32=True):
    """Random image + random cloud around the camera's forward axis (some points behind / outside the image)."""
    rng = np.random.default_rng(seed)
    intr, dist, (W, H) = CAMERAS[model]
    if size is not None:
        W, H = size
    image = rng.integers(0, 256, (H, W), dtype=np.uint8)
    # directions: mostly in front of the camera (LiDAR +x), 15 % anywhere on the sphere
    n_any = int(0.15 * n)
    d_front = S.lidar_directions("frustum", n - n_any, rng)
    d_any = S.lidar_directions("sphere", n_any, rng)
    dirs = np.concatenate([d_front, d_any])
    rng.shuffle(dirs)
    pts = dirs * rng.uniform(0.5, 25.0, (n, 1))
    if f32:
        pts = pts.astype(np.float32).astype(np.float64)
        inten = rng.integers(0, 256, n) / 256.0
    else:
        inten = rng.uniform(0.0, 1.0, n)
    xyzw = np.concatenate([pts, np.ones((n, 1))], axis=1)
    return {"model": model, "intrinsics": intr, "distortion": dist, "W": W, "H": H, "image": image, "points": xyzw, "intensities": inten, "T": S.gt_T_camera_lidar()}


def random_poses(T, count, seed=0, rot_deg=2.0, trans=0.1):
    rng = np.random.default_rng(seed)
    out = [T]
    for _ in range(count - 1):
        out.append(S.perturb(T, rng.uniform(-rot_deg, rot_deg, 3), rng.uniform(-trans, trans, 3)))
    return np.stack(out)


def digest(a):
    """SHA-256 of an array's shape and bits (floats as float64 with every NaN as one bit pattern, integers as int64): a
    bit-exact comparison with an output too large to store.  Signed zeros and infinities count."""
    a = np.asarray(a)
    a = a.astype(np.float64) if a.dtype.kind == "f" else a.astype(np.int64)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def plain(x):
    """numpy values -> JSON values (float64 round-trips exactly through json's repr of floats)."""
    if isinstance(x, dict):
        return {k: plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [plain(v) for v in x]
    if isinstance(x, np.ndarray):
        return plain(x.tolist())
    if isinstance(x, (bool, np.bool_)):
        return bool(x)
    if isinstance(x, (int, np.integer)):
        return int(x)
    if isinstance(x, (float, np.floating)):
        return float(x)
    return x


def reference_outputs():
    """What the reference's own code returned on the seeded inputs of the reference comparisons
    (tests/golden/make_reference_outputs.py)."""
    with open(REFERENCE_OUTPUTS) as f:
        return json.load(f)


def same(a, b):
    """Bit-for-bit equality of stored and computed values, NaN equal to NaN."""
    return digest(a) == digest(b)
