"""The CUDA path against the REFERENCE's own code, directly: what the reference's sources of the path (compiled against
stand-in third-party headers, oracle/ref_shim.cpp -> oracle/_ref/libvlcal_ref.so) return on the problems below is stored in
tests/golden/reference_outputs.json (tests/golden/make_reference_outputs.py).  Everything here is also implied by
(CUDA == oracle, tests/test_gpu_parity.py) and (oracle == reference, tests/test_reference_pin.py); this file closes the
triangle without the oracle in between.

`reference_side(R, pr)` computes the reference's answers; a CPU test checks the stored answers against the oracle so that
the GPU test cannot fail (or pass) because of a mistake in the helper."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import util

NID_TOL = 1e-12


def _problem(model="plumb_bob"):
    from direct_visual_lidar_calibration_b200 import synthetic as S

    if model == "plumb_bob":
        bag = S.make_bag("pinhole_640x480", "frustum", 30000, config_index=21, scale=0.5)
        T_init = S.perturb(bag["T_gt"], (0.3, -0.3, 0.3), (0.01, -0.01, 0.01))
        return {"model": bag["camera_model"], "intrinsics": bag["intrinsics"], "distortion": bag["distortion"], "W": bag["width"], "H": bag["height"], "image": bag["image"],
                "points": bag["points"], "intensities": bag["intensities"], "T": T_init}
    return util.random_problem(model, n=20000, seed=31)


def _sophus_params(T):
    return np.concatenate([Rotation.from_matrix(T[:3, :3]).as_quat(), T[:3, 3]])


def _poses(pr):
    return util.random_poses(pr["T"], 3, seed=17, rot_deg=1.0, trans=0.05)


MODELS = ["plumb_bob", "fisheye", "equirectangular"]


def reference_side(R, pr, inner_iterations=40):
    """What the reference's code returns for this problem (mode A NID at 3 poses, culling, mode B value + gradient; on the
    pinhole scene also one inner Nelder-Mead solve and a two-iteration outer loop)."""
    rc = R.Camera(pr["model"], pr["intrinsics"], pr["distortion"])
    Ts = _poses(pr)
    bags = [(pr["image"], pr["points"], pr["intensities"])]
    out = {"fov": R.estimate_camera_fov(rc, pr["W"], pr["H"]), "nid": R.nid_calculate(rc, pr["image"], pr["points"], pr["intensities"], 16, Ts),
           "cull": util.digest(R.view_cull(rc, pr["W"], pr["H"], True, pr["points"], pr["T"]))}
    sub = slice(0, 5000)
    out["modeb"] = R.nid_cost_bspline_jet(rc, pr["image"], pr["points"][sub], pr["intensities"][sub], 16, _sophus_params(pr["T"]))
    if pr["model"] == "plumb_bob":
        inner = R.calibrate_nelder_mead(rc, bags, pr["T"], max_outer_iterations=1, max_inner_iterations=inner_iterations)
        out["inner"] = {k: inner[k] for k in ("T", "num_callbacks", "callback_T")}
        out["outer"] = {"T": R.calibrate_nelder_mead(rc, bags, pr["T"], max_outer_iterations=2, max_inner_iterations=inner_iterations, delta_trans_thresh=1e-9, delta_rot_thresh=1e-9)["T"]}
    return out


def reference_outputs(R):
    return {f"gpu_triangle/{model}": reference_side(R, _problem(model)) for model in MODELS}


def _stored(model):
    ref = util.reference_outputs()[f"gpu_triangle/{model}"]
    ref["nid"] = np.array(ref["nid"])
    ref["modeb"][2] = np.array(ref["modeb"][2])
    if "inner" in ref:
        ref["inner"]["T"] = np.array(ref["inner"]["T"])
        ref["inner"]["callback_T"] = np.array(ref["inner"]["callback_T"]).reshape(-1, 4, 4)
        ref["outer"]["T"] = np.array(ref["outer"]["T"])
    return ref


def test_reference_side_helper_agrees_with_the_oracle(oracle):
    pr = _problem()
    ref = _stored("plumb_bob")
    O = oracle
    cam = O.create_camera(pr["model"], pr["intrinsics"], pr["distortion"])
    fov = O.estimate_camera_fov(cam, pr["W"], pr["H"])
    assert fov == ref["fov"]
    assert np.array_equal([O.nid_calculate(cam, pr["image"], pr["points"], pr["intensities"], 16, fov, T)[0] for T in _poses(pr)], ref["nid"])
    assert util.digest(O.view_cull(cam, pr["W"], pr["H"], fov, True, pr["points"], pr["T"])) == ref["cull"]
    p = O.default_calib_params()
    p.max_inner_iterations, p.max_outer_iterations = 40, 1
    bags = [(pr["image"], pr["points"], pr["intensities"])]
    assert np.array_equal(O.estimate_pose_nelder_mead(cam, bags, pr["T"], p)["T"], ref["inner"]["T"])
    p.max_outer_iterations, p.delta_trans_thresh, p.delta_rot_thresh = 2, 1e-9, 1e-9
    assert np.array_equal(O.calibrate(cam, bags, pr["T"], p)["T"], ref["outer"]["T"])
    ok, nid, grad = O.nid_cost_bspline_grad(cam, pr["image"], pr["points"][:5000], pr["intensities"][:5000], 16, _sophus_params(pr["T"]))
    assert [ok, nid] == ref["modeb"][:2] and np.array_equal(grad, ref["modeb"][2])


@pytest.mark.gpu
@pytest.mark.parametrize("model", MODELS)
def test_cuda_path_equals_the_reference_build(gpu, model):
    V = gpu
    pr = _problem(model)
    ref = _stored(model)
    cam = V.create_camera(pr["model"], pr["intrinsics"], pr["distortion"])
    data = V.VisualLiDARData(pr["image"], pr["points"], pr["intensities"])
    cost = V.CostCalculatorNID(cam, data)
    assert cost.max_fov == ref["fov"]
    nid = cost.calculate_batch(_poses(pr))
    assert np.all(np.abs(nid - ref["nid"]) < NID_TOL), np.abs(nid - ref["nid"]).max()
    assert util.digest(V.ViewCulling(cam, (pr["W"], pr["H"])).cull_indices(pr["points"], pr["T"])) == ref["cull"]
    # mode B: value and the 7 partials of the reference functor instantiated with Jets
    ok_r, nid_r, grad_r = ref["modeb"]
    nc = V.NIDCost(cam, V.VisualLiDARData(pr["image"], pr["points"][:5000], pr["intensities"][:5000]), 16)
    ok, nid_b, grad = nc.evaluate_with_gradient(_sophus_params(pr["T"])[None])
    assert bool(ok[0]) == ok_r and abs(nid_b[0] - nid_r) < 1e-9 and np.abs(grad[0] - grad_r).max() < 1e-8 * max(1.0, np.abs(grad_r).max())
    if model != "plumb_bob":
        return  # the solves below replay thousands of comparisons of NID values; they are pinned on the pinhole scene
    # inner solve and outer loop: identical decisions -> identical pose, same number of best-cost callbacks
    params = V.VisualCameraCalibrationParams()
    params.max_inner_iterations = 40
    calib = V.VisualCameraCalibration(cam, [data], params)
    T, r = calib.estimate_pose_nelder_mead(pr["T"])
    assert np.abs(T - ref["inner"]["T"]).max() == 0.0 and len(calib.trace) == ref["inner"]["num_callbacks"]
    for (Tg, _), Tr in zip(calib.trace, ref["inner"]["callback_T"]):
        assert np.abs(Tg - Tr).max() == 0.0
    params.max_outer_iterations, params.delta_trans_thresh, params.delta_rot_thresh = 2, 1e-9, 1e-9
    T2 = V.VisualCameraCalibration(cam, [data], params).calibrate(pr["T"])
    assert np.abs(T2 - ref["outer"]["T"]).max() < 1e-15
