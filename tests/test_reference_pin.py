"""Pins the oracle (oracle/vlcal_oracle.c) against the REFERENCE's own sources of the path (oracle/ref_shim.cpp +
oracle/ref_standin/ -> oracle/_ref/libvlcal_ref.so).

What runs on the reference side is the reference's code: create_camera.cpp + camera/*.hpp, dfo/nelder_mead.hpp,
estimate_fov.cpp, cost_calculator_nid.cpp, view_culling.cpp.  Third-party headers (Eigen, cv::Mat, ...) are stand-ins,
so Eigen's own reduction orders are restated, not pinned (oracle/ref_standin/Eigen/Core lists the conventions); the
comparisons below are therefore bit-exact, and the NID tolerance of the GPU tests (1e-12 on the entropy tail) covers
what the stand-in cannot pin.

`reference_outputs(R)` computes the reference's side of every comparison; tests/golden/make_reference_outputs.py stores
it in tests/golden/reference_outputs.json (an output too large to store is kept as a SHA-256 of its bits, util.digest),
and the tests compare the oracle with that file, so they need neither the reference tree nor its build.  CPU-only."""
import glob
import os

import numpy as np
import pytest

import util as U
from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def ref():
    return U.reference_outputs()


def cameras(model):
    intr, dist, (W, H) = U.CAMERAS[model]
    return O.create_camera(model, intr, dist), W, H


def special_points():
    e = 1e-300
    return np.array(
        [[0, 0, 0], [0, 0, 1], [0, 0, -1], [1, 0, 0], [0, 1, 0], [0, -1, 0], [1e-4, 0, 1e-4], [0, 1e-2, 1e-2], [3, 4, 1e-9], [1e-3, 1e-3, 1.0], [e, e, e], [1e200, 1e200, 1e200],
         [np.nan, 0, 1], [np.inf, 0, 1], [0.5, -0.25, 2.0], [-7.0, 3.0, 0.1], [2.0, 2.0, -0.5], [0.0, 0.0, 1e-320]], dtype=np.float64)


def projection_points():
    rng = np.random.default_rng(11)
    return np.concatenate([rng.normal(size=(30000, 3)) * rng.uniform(0.01, 40.0, (30000, 1)), special_points()])


PADDING_DISTORTIONS = ([], [-0.04], [-0.04, 0.08, 1e-4, -3e-4, -0.04, 9.0, 9.0])  # zero-padded / truncated (create_camera.cpp:24-27)


def _objectives():
    def rosenbrock(x):
        return float(100.0 * (x[1] - x[0] ** 2) ** 2 + (1.0 - x[0]) ** 2)

    def bowl(x):
        return float(np.sum((x - np.arange(len(x)) * 0.1) ** 2))

    def plateau(x):  # many exact ties: the sort / comparison order decides the trajectory
        return float(np.floor(4.0 * np.abs(x).sum()) / 4.0)

    def with_nan(x):  # NaN scores take the reference's comparison path
        return float("nan") if x[0] > 0.15 else float(np.sum(x * x) + np.sin(5.0 * x[-1]))

    def ridge(x):
        return float(abs(x[0] - x[1]) + 0.01 * np.sum(x * x))

    return {"rosenbrock": rosenbrock, "bowl": bowl, "plateau": plateau, "with_nan": with_nan, "ridge": ridge}


def nelder_mead_trials(n):
    rng = np.random.default_rng(5 + n)
    for trial, kw in enumerate([dict(), dict(init_step=1e-3, convergence_var_thresh=1e-10, max_iterations=60), dict(init_step=0.5, max_iterations=7)]):
        yield (rng.uniform(-0.3, 0.3, n) if trial else np.zeros(n)), kw


def nelder_mead_summary(r):
    """A Nelder-Mead run as stored: every objective call in order (digest), the result fields."""
    calls = np.array([np.append(x, y) for x, y in r["calls"]])
    return {"num_calls": len(r["calls"]), "calls": U.digest(calls), "converged": bool(r["converged"]), "num_iterations": int(r["num_iterations"]), "x": r["x"], "y": r["y"]}


def nid_problem(model, bins):
    pr = U.random_problem(model, n=30000, seed=21, f32=(bins == 16))
    return pr, U.random_poses(pr["T"], 4, seed=3)


def edge_case_inputs():
    """(points, intensities) of the NID edge cases: every point behind the camera (no inliers -> 0/0 -> NaN,
    cost_calculator_nid.cpp:54-57); intensities outside [0, 1), NaN intensities, NaN / huge coordinates; one point."""
    pr = U.random_problem("plumb_bob", n=2000, seed=2)
    behind = pr["points"].copy()
    behind[:, 0] = -np.abs(behind[:, 0]) - 1.0
    ins = pr["intensities"].copy()
    ins[::7] = 1.0
    ins[1::7] = -0.5
    ins[2::7] = 3.0
    ins[3::97] = np.nan
    pts = pr["points"].copy()
    pts[5::211, 1] = np.nan
    pts[6::211, 2] = 1e30
    return pr, [(behind, pr["intensities"]), (pts, ins), (pr["points"][:1], pr["intensities"][:1])]


def _sophus_params(T):
    from scipy.spatial.transform import Rotation

    q = Rotation.from_matrix(T[:3, :3]).as_quat()  # x y z w
    return np.concatenate([q, T[:3, 3]])


def bspline_cases(model):
    pr = U.random_problem(model, n=8000, seed=71)
    return pr, [(bins, _sophus_params(T)) for bins, T in zip((16, 16, 8), U.random_poses(pr["T"], 3, seed=5))]


def bspline_failure_inputs():
    pr = U.random_problem("plumb_bob", n=100, seed=72)
    far = np.array([[1.0, 5e3, 0.0, 1.0]] * 10)  # far off to the side: every projection lands outside the image
    return pr, far, np.full(10, 0.5), _sophus_params(pr["T"])


def estimate_pose_inputs(model, n_bags):
    bags = []
    for b in range(n_bags):
        pr = U.random_problem(model, n=6000 + 500 * b, seed=90 + b)
        bags.append((pr["image"], pr["points"], pr["intensities"]))
    return bags, U.random_poses(pr["T"], 1, seed=12, rot_deg=0.5, trans=0.02)[0]


ESTIMATE_POSE_CASES = [("plumb_bob", 1), ("plumb_bob", 2), ("fisheye", 1), ("equirectangular", 2)]
OUTER_LOOP_SETTINGS = (dict(max_outer_iterations=3, max_inner_iterations=25, delta_trans_thresh=1e-9, delta_rot_thresh=1e-9),  # never converges: 3 outer iterations
                       dict(max_outer_iterations=5, max_inner_iterations=25),  # default thresholds: stops after the first
                       dict(max_outer_iterations=2, max_inner_iterations=30, disable_z_buffer_culling=True, nelder_mead_init_step=5e-3))


def outer_loop_inputs():
    pr = U.random_problem("plumb_bob", n=8000, seed=95)
    return [(pr["image"], pr["points"], pr["intensities"])], U.random_poses(pr["T"], 1, seed=13, rot_deg=0.5, trans=0.02)[0]


def gradient_cases(model):
    pr = U.random_problem(model, n=6000, seed=75)
    return pr, [(bins, _sophus_params(T)) for bins, T in zip((16, 8), U.random_poses(pr["T"], 2, seed=6))]


def smooth_image_inputs():
    """A smooth image for the finite-difference check, and the parameter vectors of the central differences
    (row 2k: +1e-6 on parameter k, row 2k+1: -1e-6)."""
    intr, dist, (W, H) = U.CAMERAS["fisheye"]
    pr = U.random_problem("fisheye", n=6000, seed=76)
    yy, xx = np.mgrid[0:H, 0:W]
    img = (127 + 100 * np.sin(xx / 37.0) * np.cos(yy / 23.0)).astype(np.uint8)
    tp = _sophus_params(pr["T"])
    steps = []
    for k in range(7):
        a, b = tp.copy(), tp.copy()
        a[k] += 1e-6
        b[k] -= 1e-6
        steps += [a, b]
    return pr, img, tp, steps


def _random_camera(model, rng):
    W, H = int(rng.integers(64, 400)), int(rng.integers(48, 300))
    f = rng.uniform(0.4, 1.6) * W
    intr = [f, f * rng.uniform(0.9, 1.1), W * rng.uniform(0.4, 0.6), H * rng.uniform(0.4, 0.6)]
    if model == "plumb_bob":
        dist = list(rng.normal(0, [0.05, 0.05, 1e-3, 1e-3, 0.02]))
    elif model == "fisheye":
        dist = list(rng.normal(0, [0.02, 0.01, 0.005, 0.002]))
    elif model == "atan":
        dist = [float(rng.choice([0.0, 1e-8, rng.uniform(0.2, 1.2)]))]  # includes the d0 < 1e-7 branch (atan.hpp:17)
    elif model == "omnidir":
        intr = intr + [rng.uniform(0.5, 1.5)]
        dist = list(rng.normal(0, [0.05, 0.02, 1e-3, 1e-3]))
    elif model == "equirectangular":
        intr, dist = [float(W), float(H)], []
    else:
        dist = list(rng.normal(0, [0.05, 0.05, 1e-3, 1e-3, 0.02, 0.05, 0.03, 0.01]))
    return intr, dist, W, H


def fuzz_cases(model):
    """Random intrinsics / distortions / image sizes, with the cloud, poses and bin count of each trial."""
    rng = np.random.default_rng(1000 + U.MODELS.index(model))
    for trial in range(8):
        intr, dist, W, H = _random_camera(model, rng)
        pts = rng.normal(size=(3000, 3)) * rng.uniform(0.05, 30.0, (3000, 1))
        pr = U.random_problem(model, n=4000, seed=2000 + trial, size=(W, H))
        Ts = U.random_poses(pr["T"], 2, seed=trial, rot_deg=4.0, trans=0.3)
        bins = int(rng.choice([4, 16, 64]))
        yield intr, dist, W, H, pts, pr, Ts, bins


def lidar_image_inputs(model):
    pr = U.random_problem(model, n=30000, seed=5)
    pts = np.concatenate([pr["points"], pr["points"][:2000]])  # exact duplicates: equal squared ranges
    ins = np.concatenate([pr["intensities"], (pr["intensities"][:2000] + 0.5) % 1.0])
    return pr, pts, ins


def golden_files(mode):
    files = sorted(glob.glob(os.path.join(HERE, "golden", f"mode_{mode}_*.npz")))
    assert len(files) == len(U.MODELS)
    return [(os.path.basename(p)[len(f"mode_{mode}_"):-len(".npz")], np.load(p)) for p in files]


def reference_outputs(R):
    """The reference's side of every comparison below, from its own code (R = oracle.reference, which needs
    oracle/_ref/libvlcal_ref.so)."""
    out = {}
    for model in U.MODELS:
        intr, dist, (W, H) = U.CAMERAS[model]
        rc = R.Camera(model, intr, dist)
        out[f"project/{model}"] = U.digest(R.project(rc, projection_points()))
        out[f"fov/{model}"] = [R.estimate_camera_fov(rc, W, H), R.estimate_camera_fov(rc, W // 2 + 1, H // 3)]
        for bins in (16, 8):
            pr, Ts = nid_problem(model, bins)
            out[f"nid/{model}/{bins}"] = R.nid_calculate(rc, pr["image"], pr["points"], pr["intensities"], bins, Ts)
        pr = U.random_problem(model, n=40000, seed=33)
        for depth in (True, False):
            out[f"cull/{model}/{depth}"] = [U.digest(R.view_cull(rc, W, H, depth, pr["points"], T)) for T in U.random_poses(pr["T"], 2, seed=8)]
        pr, cases = bspline_cases(model)
        out[f"bspline/{model}"] = [R.nid_cost_bspline(rc, pr["image"], pr["points"], pr["intensities"], bins, tp) for bins, tp in cases]
        pr, cases = gradient_cases(model)
        out[f"bspline_grad/{model}"] = [R.nid_cost_bspline_jet(rc, pr["image"], pr["points"], pr["intensities"], bins, tp) for bins, tp in cases]
        fuzz = []
        for intr_f, dist_f, Wf, Hf, pts, pr, Ts, bins in fuzz_cases(model):
            rf = R.Camera(model, intr_f, dist_f)
            fuzz.append({"project": U.digest(R.project(rf, pts)), "fov": R.estimate_camera_fov(rf, Wf, Hf), "nid": R.nid_calculate(rf, pr["image"], pr["points"], pr["intensities"], bins, Ts),
                         "cull": U.digest(R.view_cull(rf, Wf, Hf, True, pr["points"], Ts[0]))})
        out[f"fuzz/{model}"] = fuzz
        pr, pts, ins = lidar_image_inputs(model)
        inten, index = R.generate_lidar_image(R.Camera(model, pr["intrinsics"], pr["distortion"]), pr["W"], pr["H"], pr["T"], pts, ins)
        out[f"lidar_image/{model}"] = {"intensity": U.digest(inten), "index": U.digest(index)}

    out["camera_rejected"] = [R.Camera("no_such_model", [1, 1, 1, 1], []).handle is None, R.Camera("plumb_bob", [1, 1, 1], []).handle is None]
    out["camera_padding"] = [R.project(R.Camera("plumb_bob", [400, 410, 320, 240], d), np.array([[0.3, -0.2, 1.5]]))[0] for d in PADDING_DISTORTIONS]
    for n in (2, 3, 6):
        for name, f in _objectives().items():
            out[f"nelder_mead/{name}/{n}"] = [nelder_mead_summary(R.nelder_mead(f, x0, **kw)) for x0, kw in nelder_mead_trials(n)]

    rc = R.Camera("plumb_bob", *U.CAMERAS["plumb_bob"][:2])
    pr, cases = edge_case_inputs()
    out["nid_edge"] = [R.nid_calculate(rc, pr["image"], pts, ins, 16, [pr["T"]])[0] for pts, ins in cases]
    pr, far, ins, tp = bspline_failure_inputs()
    out["bspline_failure_ok"] = R.nid_cost_bspline(rc, pr["image"], far, ins, 16, tp)[0]
    bags, T0 = outer_loop_inputs()
    out["calibrate_outer"] = [R.calibrate_nelder_mead(rc, bags, T0, **kw)["T"] for kw in OUTER_LOOP_SETTINGS]
    for model, n_bags in ESTIMATE_POSE_CASES:
        bags, T0 = estimate_pose_inputs(model, n_bags)
        r = R.calibrate_nelder_mead(R.Camera(model, *U.CAMERAS[model][:2]), bags, T0, max_outer_iterations=1, max_inner_iterations=40)
        out[f"estimate_pose/{model}/{n_bags}"] = {"T": r["T"], "num_callbacks": r["num_callbacks"], "callback_T": U.digest(r["callback_T"])}
    rf = R.Camera("fisheye", *U.CAMERAS["fisheye"][:2])
    pr, img, _, steps = smooth_image_inputs()
    out["bspline_fd"] = [R.nid_cost_bspline(rf, img, pr["points"], pr["intensities"], 16, t)[1] for t in steps]

    for model, g in golden_files("a"):
        H, W = g["image"].shape
        rg = R.Camera(model, g["intrinsics"], g["distortion"])
        pts, ins = g["points"].astype(np.float64), g["intensities"].astype(np.float64)
        out[f"golden_mode_a/{model}"] = {"max_fov": R.estimate_camera_fov(rg, W, H), "nid": R.nid_calculate(rg, g["image"], pts, ins, 16, g["poses"]),
                                         "cull_indices": U.digest(R.view_cull(rg, W, H, True, pts, g["poses"][0]))}
    for model, g in golden_files("b"):
        rg = R.Camera(model, g["intrinsics"], g["distortion"])
        pts, ins = g["points"].astype(np.float64), g["intensities"].astype(np.float64)
        out[f"golden_mode_b/{model}"] = [{"jet": R.nid_cost_bspline_jet(rg, g["image"], pts, ins, 16, tp), "double": R.nid_cost_bspline(rg, g["image"], pts, ins, 16, tp)[1]}
                                         for tp in g["T_params"]]
    return out


@pytest.mark.parametrize("model", U.MODELS)
def test_projection_bit_exact(ref, model):
    oc, W, H = cameras(model)
    uv_o = np.array([O.project(oc, p) for p in projection_points()])
    assert U.digest(uv_o) == ref[f"project/{model}"]  # every bit, signed zeros included


def test_create_camera_rejections(ref):
    assert ref["camera_rejected"] == [True, True]  # create_camera.cpp:49-50, :19-22
    assert O.create_camera("no_such_model", [1, 1, 1, 1], []) is None
    assert O.create_camera("plumb_bob", [1, 1, 1], []) is None
    for dist, want in zip(PADDING_DISTORTIONS, ref["camera_padding"]):
        oc = O.create_camera("plumb_bob", [400, 410, 320, 240], dist)
        assert np.array_equal(O.project(oc, np.array([0.3, -0.2, 1.5])), want)


@pytest.mark.parametrize("model", U.MODELS)
def test_estimate_camera_fov_bit_exact(ref, model):
    oc, W, H = cameras(model)
    assert O.estimate_camera_fov(oc, W, H) == ref[f"fov/{model}"][0]
    assert O.estimate_camera_fov(oc, W // 2 + 1, H // 3) == ref[f"fov/{model}"][1]  # odd sizes: integer halves (:37)


@pytest.mark.parametrize("n", [2, 3, 6])
@pytest.mark.parametrize("name", list(_objectives().keys()))
def test_nelder_mead_trajectory_identical(ref, n, name):
    f = _objectives()[name]
    for trial, ((x0, kw), b) in enumerate(zip(nelder_mead_trials(n), ref[f"nelder_mead/{name}/{n}"])):
        a = nelder_mead_summary(O.nelder_mead(f, x0, **kw))
        assert a["num_calls"] == b["num_calls"] and a["calls"] == b["calls"], (name, n, trial)
        assert a["converged"] == b["converged"] and a["num_iterations"] == b["num_iterations"]
        assert U.same(a["x"], b["x"]) and U.same(a["y"], b["y"])


@pytest.mark.parametrize("model", U.MODELS)
@pytest.mark.parametrize("bins", [16, 8])
def test_nid_calculate_bit_exact(ref, model, bins):
    oc, W, H = cameras(model)
    fov = O.estimate_camera_fov(oc, W, H)
    pr, Ts = nid_problem(model, bins)
    want = np.array([O.nid_calculate(oc, pr["image"], pr["points"], pr["intensities"], bins, fov, T)[0] for T in Ts])
    assert U.same(ref[f"nid/{model}/{bins}"], want), (ref[f"nid/{model}/{bins}"], want)


def test_nid_calculate_edge_cases(ref):
    oc, W, H = cameras("plumb_bob")
    fov = O.estimate_camera_fov(oc, W, H)
    pr, cases = edge_case_inputs()
    got = [O.nid_calculate(oc, pr["image"], pts, ins, 16, fov, pr["T"])[0] for pts, ins in cases]
    assert np.isnan(got[0]) and np.isnan(ref["nid_edge"][0])  # no inliers: NaN on both sides
    assert got[1] == ref["nid_edge"][1]
    assert U.same(got[2], ref["nid_edge"][2])  # a single point


@pytest.mark.parametrize("model", U.MODELS)
@pytest.mark.parametrize("depth", [True, False])
def test_view_culling_indices_identical(ref, model, depth):
    oc, W, H = cameras(model)
    fov = O.estimate_camera_fov(oc, W, H)
    pr = U.random_problem(model, n=40000, seed=33)
    for T, want in zip(U.random_poses(pr["T"], 2, seed=8), ref[f"cull/{model}/{depth}"]):
        assert U.digest(O.view_cull(oc, W, H, fov, depth, pr["points"], T)) == want


def test_golden_fixtures_match_the_reference(ref):
    """The committed fixtures (made from the oracle, tests/golden/make_golden.py) are what the reference's code returns."""
    for model, g in golden_files("a"):
        want = ref[f"golden_mode_a/{model}"]
        assert float(g["max_fov"]) == want["max_fov"]
        assert U.same(g["nid"], want["nid"])
        assert U.digest(g["cull_indices"]) == want["cull_indices"]


@pytest.mark.parametrize("model", U.MODELS)
def test_bspline_nid_value_bit_exact(ref, model):
    """NIDCost::operator()<double> (include/vlcal/costs/nid_cost.hpp:36-107), the value half of the BFGS branch."""
    oc, W, H = cameras(model)
    pr, cases = bspline_cases(model)
    for (bins, tp), (ok_r, nid_r) in zip(cases, ref[f"bspline/{model}"]):
        ok_o, nid_o, _ = O.nid_cost_bspline(oc, pr["image"], pr["points"], pr["intensities"], bins, tp)
        assert ok_r and ok_o and nid_r == nid_o, (nid_r, nid_o)


def test_bspline_failure_flag(ref):
    oc, W, H = cameras("plumb_bob")
    pr, far, ins, tp = bspline_failure_inputs()
    ok_o, _, _ = O.nid_cost_bspline(oc, pr["image"], far, ins, 16, tp)
    assert ref["bspline_failure_ok"] is False and ok_o is False  # no inliers -> NaN -> the functor returns false (nid_cost.hpp:98-102)


def _best_cost_poses(init_T, trace):
    """Poses the reference hands to params.callback: evaluations that improve on the best cost so far (:112-116)."""
    best, out = np.finfo(np.float64).max, []
    for row in trace:
        if row[6] < best:
            best = row[6]
            out.append(O.isometry_mul(init_T, O.se3_expmap(row[:6])))
    return out


@pytest.mark.parametrize("model,n_bags", ESTIMATE_POSE_CASES)
def test_estimate_pose_nelder_mead_identical(ref, model, n_bags):
    """VisualCameraCalibration::estimate_pose_nelder_mead (visual_camera_calibration.cpp:70-139) through calibrate() with
    one outer iteration: culling at the start pose, one cost object per bag, objective sum in bag order, best-cost
    callbacks, result init_T * Expmap(x).  (GTSAM's Expmap and Eigen's Isometry product are stand-ins on the reference
    side -- restated like the oracle's; everything else is the reference's code.)"""
    oc, W, H = cameras(model)
    bags, T0 = estimate_pose_inputs(model, n_bags)
    p = O.default_calib_params()
    p.max_inner_iterations = 40
    p.max_outer_iterations = 1
    a = O.estimate_pose_nelder_mead(oc, bags, T0, p)
    b = ref[f"estimate_pose/{model}/{n_bags}"]
    assert U.same(a["T"], b["T"])
    want = _best_cost_poses(T0, a["trace"])
    assert b["num_callbacks"] == len(want)
    assert U.digest(np.array(want).reshape(len(want), 4, 4)) == b["callback_T"]


def test_calibrate_outer_loop_identical(ref):
    """VisualCameraCalibration::calibrate (visual_camera_calibration.cpp:35-68): re-culling at every outer iteration and
    the delta_t / delta_r termination test."""
    oc, W, H = cameras("plumb_bob")
    bags, T0 = outer_loop_inputs()
    for kw, want in zip(OUTER_LOOP_SETTINGS, ref["calibrate_outer"]):
        p = O.default_calib_params()
        p.max_outer_iterations, p.max_inner_iterations = kw["max_outer_iterations"], kw["max_inner_iterations"]
        p.delta_trans_thresh = kw.get("delta_trans_thresh", p.delta_trans_thresh)
        p.delta_rot_thresh = kw.get("delta_rot_thresh", p.delta_rot_thresh)
        p.disable_z_buffer_culling = int(kw.get("disable_z_buffer_culling", False))
        p.nelder_mead_init_step = kw.get("nelder_mead_init_step", p.nelder_mead_init_step)
        a = O.calibrate(oc, bags, T0, p)
        assert U.same(a["T"], want), kw


@pytest.mark.parametrize("model", U.MODELS)
def test_bspline_nid_gradient_bit_exact(ref, model):
    """NIDCost::operator()<ceres::Jet<double, 7>> (what AutoDiffFirstOrderFunction evaluates in the BFGS branch,
    visual_camera_calibration.cpp:211): residual and its 7 partials, reference functor + stand-in Jet vs the oracle."""
    oc, W, H = cameras(model)
    pr, cases = gradient_cases(model)
    for (bins, tp), (ok_r, nid_r, g_r) in zip(cases, ref[f"bspline_grad/{model}"]):
        ok_o, nid_o, g_o = O.nid_cost_bspline_grad(oc, pr["image"], pr["points"], pr["intensities"], bins, tp)
        assert ok_r and ok_o and nid_r == nid_o and U.same(g_r, g_o), (nid_r, nid_o, g_r, g_o)
        assert np.abs(g_o).max() > 1e-4


def test_bspline_gradient_is_the_derivative_of_the_value(ref):
    """Independent of any Jet arithmetic: central differences of the reference's double functor on a smooth image."""
    oc, W, H = cameras("fisheye")
    pr, img, tp, _ = smooth_image_inputs()
    _, _, g = O.nid_cost_bspline_grad(oc, img, pr["points"], pr["intensities"], 16, tp)
    vals = np.array(ref["bspline_fd"])
    fd = (vals[0::2] - vals[1::2]) / 2e-6
    assert np.abs(g - fd).max() < 1e-5 * max(1.0, np.abs(g).max()), (g, fd)


@pytest.mark.parametrize("model", U.MODELS)
def test_fuzz_random_cameras_projection_fov_nid_culling(ref, model):
    """Random intrinsics / distortions / image sizes (the fixed presets above could hide a branch): projection, FoV, NID and
    culling of the oracle against the reference's code, bit for bit."""
    for trial, ((intr, dist, W, H, pts, pr, Ts, bins), want) in enumerate(zip(fuzz_cases(model), ref[f"fuzz/{model}"])):
        oc = O.create_camera(model, intr, dist)
        assert U.digest(np.array([O.project(oc, p) for p in pts])) == want["project"], (model, trial)
        fov = O.estimate_camera_fov(oc, W, H)
        assert fov == want["fov"], (model, trial, intr, dist)
        got = np.array([O.nid_calculate(oc, pr["image"], pr["points"], pr["intensities"], bins, fov, T)[0] for T in Ts])
        assert U.same(got, want["nid"]), (model, trial, got, want["nid"])
        assert U.digest(O.view_cull(oc, W, H, fov, True, pr["points"], Ts[0])) == want["cull"]


def test_mode_b_golden_fixtures_match_reference_and_oracle(ref):
    """tests/golden/mode_b_*.npz were written from the reference functor (make_golden.py); the reference's values and the
    oracle must reproduce them exactly."""
    for model, g in golden_files("b"):
        oc = O.create_camera(model, g["intrinsics"], g["distortion"])
        pts, ins = g["points"].astype(np.float64), g["intensities"].astype(np.float64)
        for k, (tp, want) in enumerate(zip(g["T_params"], ref[f"golden_mode_b/{model}"])):
            ok_r, nid_r, grad_r = want["jet"]
            ok_o, nid_o, grad_o = O.nid_cost_bspline_grad(oc, g["image"], pts, ins, 16, tp)
            assert ok_r and ok_o and nid_r == nid_o == g["nid_jet_functor"][k]
            assert U.same(grad_r, g["grad"][k]) and np.array_equal(grad_o, g["grad"][k])
            assert want["double"] == g["nid_double_functor"][k] == O.nid_cost_bspline(oc, g["image"], pts, ins, 16, tp)[1]


@pytest.mark.parametrize("model", U.MODELS)
def test_generate_lidar_image_equals_the_reference(ref, model):
    """generate_lidar_image (src/vlcal/preprocess/generate_lidar_image.cpp:8-41): the oracle's intensity image and index map
    equal the reference's own code bit for bit, including the tie rule (of equal squared ranges the last point wins)."""
    pr, pts, ins = lidar_image_inputs(model)
    cam = O.create_camera(model, pr["intrinsics"], pr["distortion"])
    a = O.generate_lidar_image(cam, pr["W"], pr["H"], pr["T"], pts, ins)
    assert U.digest(a[0]) == ref[f"lidar_image/{model}"]["intensity"] and U.digest(a[1]) == ref[f"lidar_image/{model}"]["index"]
    assert (a[1] >= 30000).sum() > 100  # duplicates won their pixels
