"""CPU: pin the oracle's building blocks against independent re-derivations (numpy / scipy), the
closed forms they must satisfy, and the sanity band of the reference's own test programs.

The reference itself cannot be built here (Eigen/OpenCV/Sophus/vikit absent) and its tests are
print-only programs on an external dataset, so these are the strongest pins available:
"PARITY UNPINNED" at the vikit/Sophus boundary remains stated in oracle/svo_oracle.h and DESIGN.md.
"""
import numpy as np
import pytest
from scipy.linalg import expm
from scipy.stats import norm as scipy_norm

from rpg_svo_b200 import synth
from tests.reference_outputs import sha256


def _T44(T):
    return np.vstack([T, [0, 0, 0, 1]])


@pytest.mark.parametrize("scale", [1e-12, 1e-6, 1e-2, 0.5, 3.0])
def test_se3_exp_vs_scipy_expm(oracle, scale):
    rng = np.random.default_rng(1)
    for _ in range(10):
        x = rng.normal(size=6) * scale
        tw = np.zeros((4, 4))
        tw[:3, :3] = synth.hat(x[3:])
        tw[:3, 3] = x[:3]
        assert np.allclose(_T44(oracle.se3_exp(x)), expm(tw), atol=1e-12)
        assert np.allclose(oracle.se3_exp(x), synth.se3_exp(x), atol=1e-12)


def test_se3_group_ops(oracle):
    rng = np.random.default_rng(2)
    A, B = oracle.se3_exp(rng.normal(size=6)), oracle.se3_exp(rng.normal(size=6))
    assert np.allclose(_T44(oracle.se3_mul(A, B)), _T44(A) @ _T44(B), atol=1e-13)
    assert np.allclose(_T44(oracle.se3_inv(A)), np.linalg.inv(_T44(A)), atol=1e-13)
    I = oracle.se3_mul(A, oracle.se3_inv(A))
    assert np.allclose(I, synth.se3_identity(), atol=1e-14)


def test_ldlt_solve_vs_numpy(oracle):
    rng = np.random.default_rng(3)
    for _ in range(20):
        J = rng.normal(size=(40, 6)) * rng.uniform(0.1, 100, 6)
        H, b = J.T @ J, rng.normal(size=6)
        assert np.allclose(oracle.ldlt6_solve(H, b), np.linalg.solve(H, b), rtol=1e-8)
    # Eigen's LDLT of the zero matrix solves to zero, not NaN (the n_meas == 0 corner of SparseImgAlign)
    assert np.array_equal(oracle.ldlt6_solve(np.zeros((6, 6)), np.ones(6)), np.zeros(6))


def test_half_sample_rule(oracle):
    rng = np.random.default_rng(4)
    img = rng.integers(0, 256, (51, 77), dtype=np.uint8)
    out = oracle.half_sample(img)
    assert out.shape == (25, 38)
    exp = (img[0:50:2, 0:76:2].astype(int) + img[0:50:2, 1:76:2] + img[1:50:2, 0:76:2] + img[1:50:2, 1:76:2]) // 4
    assert np.array_equal(out, exp)


def _update_seed_numpy(x, tau2, a, b, mu, z_range, sigma2):
    """Independent float32 transcription of the Vogiatzis-Hernandez update (depth_filter.cpp:309-332)."""
    f32 = np.float32
    x, tau2, a, b, mu, z_range, sigma2 = map(f32, (x, tau2, a, b, mu, z_range, sigma2))
    norm_scale = np.sqrt(sigma2 + tau2)
    s2 = f32(1.0 / (1.0 / float(sigma2) + 1.0 / float(tau2)))
    m = s2 * (mu / sigma2 + x / tau2)
    C1 = a / (a + b) * f32(scipy_norm.pdf(float(x), float(mu), float(norm_scale)))
    C2 = f32(float(b / (a + b)) / float(z_range))
    nc = C1 + C2
    C1, C2 = C1 / nc, C2 / nc
    f = f32(float(C1) * (float(a) + 1.0) / (float(a + b) + 1.0) + float(C2 * a) / (float(a + b) + 1.0))
    e = f32(float(C1) * (float(a) + 1.0) * (float(a) + 2.0) / ((float(a + b) + 1.0) * (float(a + b) + 2.0))
            + float(C2 * a * (a + f32(1)) / ((a + b + f32(1)) * (a + b + f32(2)))))
    mu_new = C1 * m + C2 * mu
    sigma2_new = C1 * (s2 + m * m) + C2 * (sigma2 + mu * mu) - mu_new * mu_new
    a_new = (e - f) / (f - e / f)
    return a_new, a_new * (f32(1) - f) / f, mu_new, sigma2_new


def test_update_seed_known_answers(oracle):
    rng = np.random.default_rng(5)
    for _ in range(200):
        a, b = rng.uniform(5, 30, 2)
        mu, z_range = rng.uniform(0.2, 1.0), 2.0
        sigma2 = rng.uniform(1e-3, 0.2)
        x, tau2 = mu + rng.normal() * 0.05, rng.uniform(1e-5, 1e-2)
        s = oracle.update_seed(x, tau2, a, b, mu, z_range, sigma2)
        ea, eb, emu, es2 = _update_seed_numpy(x, tau2, a, b, mu, z_range, sigma2)
        assert np.allclose([s[0], s[1], s[2], s[4]], [ea, eb, emu, es2], rtol=5e-4)
        assert s[3] == np.float32(z_range)
    # seed constructor constants of svo/test/test_depth_filter.cpp:128: Seed(ftr, 2.0, 0.5)
    assert np.float32(1.0) / np.float32(0.5) == 2.0 and np.isclose(np.float32(2.0) ** 2 / 36, 0.1111111, atol=1e-6)
    # NaN measurement variance leaves the seed untouched (depth_filter.cpp:312)
    s = oracle.update_seed(0.5, np.nan, 10, 10, 0.5, 2.0, 0.1)
    assert np.array_equal(s, np.array([10, 10, 0.5, 2.0, 0.1], np.float32))


def test_compute_tau_closed_form(oracle):
    rng = np.random.default_rng(6)
    for _ in range(50):
        T = oracle.se3_exp(np.concatenate([rng.normal(size=3) * 0.3, rng.normal(size=3) * 0.1]))
        f = rng.normal(size=3) * 0.2 + [0, 0, 1]
        f /= np.linalg.norm(f)
        z, ang = rng.uniform(0.5, 5), 2 * np.arctan(1 / (2 * 315.5))
        t = T[:, 3]
        a = f * z - t
        alpha = np.arccos(f @ t / np.linalg.norm(t))
        beta = np.arccos(a @ (-t) / (np.linalg.norm(t) * np.linalg.norm(a)))
        exp = np.linalg.norm(t) * np.sin(beta + ang) / np.sin(3.14159265 - alpha - beta - ang) - z  # truncated PI
        assert np.isclose(oracle.compute_tau(T, f, z, ang), exp, rtol=1e-12, atol=1e-15)


def test_align2d_reference_test_procedure(oracle):
    """Replays svo/test/test_feature_alignment.cpp:54-99 on a synthetic image: patch at (130.2,120.3),
    start offset (-1.1,-0.8), 3 iterations; its printed reference errors are 1D 0.000033 px and
    2D 0.015102 px on the Blender image -- a sanity band here, not a bit pin."""
    cam = synth.camera_for(640, 480)
    img = synth.render(cam, synth.base_pose(), synth.Plane.tilted(), synth.make_texture(7))
    px_true, px_error = np.array([130.2, 120.3]), np.array([-1.1, -0.8])
    pwb = synth.patch_with_border(img, px_true)
    ok2, p2 = oracle.align2d(img, pwb, pwb[1:9, 1:9], 3, px_true - px_error)
    ok1, p1, h_inv = oracle.align1d(img, (px_error / np.linalg.norm(px_error)).astype(np.float32), pwb, pwb[1:9, 1:9], 3,
                                    px_true - px_error)
    assert np.linalg.norm(p2 - px_true) < 0.1
    assert np.linalg.norm(p1 - px_true) < 0.05
    assert h_inv > 0
    # leaving the image -> not converged, estimate still written (quirk 9)
    ok, p = oracle.align2d(img, pwb, pwb[1:9, 1:9], 10, np.array([2.0, 2.0]))
    assert not ok and np.allclose(p, [2.0, 2.0])


def test_warp_affine_identity_and_triangulation(oracle):
    tv = synth.make_two_view(3, baseline=0.2)
    cam = tv["cam"]
    px = np.array([300.0, 260.0])  # svo/test/test_matcher.cpp:49
    f = cam.cam2world(px)
    A = oracle.warp_matrix_affine(cam, px, f, 2.0, synth.se3_identity(), 0)
    assert np.allclose(A, np.eye(2), atol=1e-9)  # no motion -> identity warp
    assert oracle.best_search_level(np.eye(2) * 2.1, 4) == 1 and oracle.best_search_level(np.eye(2), 4) == 0
    ok, patch = oracle.warp_affine(np.eye(2), tv["ref_pyr"][0], px, 0, 0, 5)
    assert ok and np.array_equal(patch, tv["ref_pyr"][0][255:265, 295:305])
    # triangulation of an exact correspondence returns the true depth
    X = synth.intersect(tv["plane"], tv["T_ref_w"], f[None])[0]
    T_cur_ref = synth.se3_mul(tv["T_cur_w"], synth.se3_inv(tv["T_ref_w"]))
    x_ref = tv["T_ref_w"][:, :3] @ X + tv["T_ref_w"][:, 3]
    x_cur = tv["T_cur_w"][:, :3] @ X + tv["T_cur_w"][:, 3]
    ok, d = oracle.depth_from_triangulation(T_cur_ref, f, x_cur / np.linalg.norm(x_cur))
    assert ok and np.isclose(d, np.linalg.norm(x_ref), rtol=1e-9)


def test_sparse_img_align_recovers_ground_truth(oracle, pair300):
    d = pair300
    r = oracle.sparse_img_align(d["ref_pyr"], d["cur_pyr"], d["cam"], synth.se3_identity(), d["px"], d["f"], d["pos"],
                                d["has_point"], d["ref_pos"], 4, 0)
    dt, dr = synth.pose_error(r["T"], d["T_cur_ref_gt"])
    assert dt < 5e-4 and dr < 5e-4
    assert r["n_tracked"] == int(d["has_point"].sum()) == int(r["visible"].sum())
    assert not np.any(r["visible"][d["has_point"] == 0])  # point == NULL never becomes visible
    # GN control flow [EXT NLLSSolver]: first iteration of a level is never rejected; a rejection ends the level
    for a, b in zip(r["trace"], r["trace"][1:]):
        if not a["accepted"]:
            assert b["level"] == a["level"] - 1 and b["iter"] == 0
    assert all(t["accepted"] for t in r["trace"] if t["iter"] == 0)
    # Fisher information is H/(5e-4*255^2): H must be symmetric positive definite
    assert np.allclose(r["H"], r["H"].T) and np.all(np.linalg.eigvalsh(r["H"]) > 0)


def test_sparse_residuals_jacobian_is_photometric_derivative(oracle, pair300):
    """The cached Jacobian column must equal d(residual)/d(xi) of the inverse-compositional model:
    finite differences of the reference-side warp, checked through Jres = -J^T r."""
    d = pair300
    T = synth.se3_identity()
    o = oracle.sparse_residuals(d["ref_pyr"][1], d["cur_pyr"][1], 1, d["cam"], T, d["px"], d["f"], d["pos"],
                                d["has_point"], d["ref_pos"])
    m = o["in_image"].astype(bool)
    J = o["jac"][m].reshape(-1, 6)
    r = o["residuals"][m].reshape(-1).astype(np.float64)
    assert np.allclose(o["H"], J.T @ J, rtol=1e-10)
    assert np.allclose(o["Jres"], -J.T @ r, rtol=1e-8, atol=1e-6)
    assert np.isclose(o["chi2"], np.mean(r ** 2), rtol=1e-5)


def test_pose_optimizer_recovers_pose(oracle):
    c = synth.make_pose_opt_case(9, 400, 752, 480, px_noise=0.0, outlier_frac=0.0)
    o = oracle.pose_optimize(2.0, 10, c["cam"].fx, c["T_init"], c["f"], c["pos"], c["level"], c["has_point"])
    dt, dr = synth.pose_error(o["T"], c["T_true"])
    assert dt < 1e-6 and dr < 1e-6
    assert o["num_obs"] == int(c["has_point"].sum()) and o["error_final"] < 1e-3
    assert np.allclose(o["cov"], o["cov"].T, rtol=1e-6)


def test_oracle_align_equals_reference_source_compiled_here(oracle, reference):
    """oracle/_ref = the reference's OWN svo/src/feature_alignment.cpp compiled in place with GCC -O3 -mfma
    (default -ffp-contract=fast) against the stand-in Eigen / cv::Mat headers in oracle/shim.  The oracle's
    restatement -- including its explicit-fma contraction pattern -- must reproduce it bit for bit."""
    c = synth.make_align_case(11, 300)
    for n_iter in (3, 10):
        for i in range(len(c["level"])):
            img = c["pyr"][c["level"][i]]
            ok_o, px_o = oracle.align2d(img, c["pwb"][i], c["patch"][i], n_iter, c["px_start"][i])
            ok_r, px_r = reference.ref_align2d(img, c["pwb"][i], c["patch"][i], n_iter, c["px_start"][i])
            assert ok_o == ok_r and np.array_equal(px_o, px_r), ("align2D", i, n_iter)
            ok_o, px_o, h_o = oracle.align1d(img, c["dir"][i], c["pwb"][i], c["patch"][i], n_iter, c["px_start"][i])
            ok_r, px_r, h_r = reference.ref_align1d(img, c["dir"][i], c["pwb"][i], c["patch"][i], n_iter, c["px_start"][i])
            assert ok_o == ok_r and np.array_equal(px_o, px_r) and h_o == h_r, ("align1D", i, n_iter)


# ---- oracle/_ref: the reference's own classes compiled from its svo/src (stand-in third-party headers); their outputs ----
# ---- on these inputs are replayed from tests/golden/reference/ (tests/reference_outputs.py) ----

@pytest.mark.parametrize("seed,levels", [(11, (4, 2)), (12, (4, 0)), (13, (2, 1))])
def test_oracle_sparse_img_align_equals_reference_source_compiled_here(oracle, seed, levels, reference):
    """svo::SparseImgAlign::run of the compiled reference (sparse_img_align.cpp + frame.cpp + config.cpp, driven by
    the stand-in vk::NLLSSolver) vs the oracle's restatement: same visibility, same reference patches bit for bit,
    same final pose."""
    p = synth.make_frame_pair(seed, n_feat=200)
    p["has_point"][::17] = 0
    r = reference.ref_sparse_img_align(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], p["cam"], p["T_ref_w"], p["T_ref_w"],
                                       p["px"], p["f"], p["pos"], p["has_point"], levels[0], levels[1])
    o = oracle.sparse_img_align(p["ref_pyr"], p["cur_pyr"], p["cam"], synth.se3_identity(), p["px"], p["f"], p["pos"],
                                p["has_point"], p["ref_pos"], levels[0], levels[1])
    T_cur_w = synth.se3_mul(o["T"], p["T_ref_w"])
    assert r["n_tracked"] == o["n_tracked"]
    assert np.array_equal(r["visible"], o["visible"])
    assert np.allclose(r["T_cur_w"], T_cur_w, rtol=0, atol=1e-9)
    assert np.allclose(r["H"], o["H"], rtol=1e-9, atol=1e-9)
    # the reference patch cache of the last level (f32 bilinear) matches the oracle's residual-stage patches
    q = oracle.sparse_residuals(p["ref_pyr"][levels[1]], p["cur_pyr"][levels[1]], levels[1], p["cam"], o["T"], p["px"],
                                p["f"], p["pos"], p["has_point"], p["ref_pos"])
    v = r["visible"].astype(bool)
    assert r["visible_ref_patch_sha256"] == sha256(q["ref_patch"][v])


@pytest.mark.parametrize("case", ["two_iterations", "five_features", "bad_initial_pose", "no_points"])
def test_oracle_sparse_img_align_corner_cases_equal_reference_source_compiled_here(oracle, case, reference):
    """svo::SparseImgAlign::run of the compiled reference at the corners of the Gauss-Newton driver: the iteration limit
    (no convergence at any level), a handful of features (H barely determined), an initial pose far enough off that updates get
    rejected (chi2 increases -> roll-back, :44-52 of the stand-in NLLSSolver), and a frame whose features have no 3D point."""
    n_feat = 5 if case == "five_features" else 200
    p = synth.make_frame_pair(77, n_feat=n_feat, trans=0.05, rot_deg=1.0)
    n_iter = 2 if case == "two_iterations" else 30
    T0 = synth.se3_identity()
    if case == "bad_initial_pose":
        T0 = synth.se3_exp(np.array([0.15, -0.12, 0.1, 0.03, -0.025, 0.02]))
    if case == "no_points":
        p["has_point"][:] = 0
    r = reference.ref_sparse_img_align(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], p["cam"], p["T_ref_w"],
                                       synth.se3_mul(T0, p["T_ref_w"]), p["px"], p["f"], p["pos"], p["has_point"], 4, 0, n_iter)
    o = oracle.sparse_img_align(p["ref_pyr"], p["cur_pyr"], p["cam"], T0, p["px"], p["f"], p["pos"], p["has_point"],
                                p["ref_pos"], 4, 0, n_iter)
    assert r["n_tracked"] == o["n_tracked"]
    assert np.array_equal(r["visible"], o["visible"])
    # T_cur_from_ref is re-formed by the reference from the two world poses: 1e-9 on the final pose, as in the main pin
    assert np.allclose(r["T_cur_w"], synth.se3_mul(o["T"], p["T_ref_w"]), rtol=0, atol=1e-8 if case == "bad_initial_pose" else 1e-9)
    if case == "two_iterations":
        assert 5 < len(o["trace"]) <= 10 and max(t["iter"] for t in o["trace"]) == 1  # the iteration limit ended the levels
    if case == "bad_initial_pose":
        assert any(not t["accepted"] for t in o["trace"])  # the roll-back path really ran
    if case == "no_points":
        assert o["n_tracked"] == 0 and np.allclose(o["T"], T0)


@pytest.mark.parametrize("level", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("camera", ["pinhole", "atan", "pinhole_radtan"])
def test_oracle_residual_pass_equals_reference_source_compiled_here(oracle, level, camera, reference):
    """svo::SparseImgAlign::computeResiduals of the compiled reference (sparse_img_align.cpp:147-243), called directly at one
    level and a perturbed pose, vs the oracle's restatement: visibility, patch cache and the magnitude of EVERY per-pixel
    residual bit for bit (the reference's `errors` vector, captured through the solver's scale estimator), chi2 / n_meas
    equal, Jres_ and H_ to rounding of the summation."""
    if camera == "pinhole":
        p = synth.make_frame_pair(1000, n_feat=300, n_levels=5)
    else:  # the parameter files the reference ships (752x480)
        cam = synth.reference_param_camera(camera)
        p = synth.make_frame_pair(1000, width=cam.width, height=cam.height, n_feat=300, n_levels=5, cam=cam)
    p["has_point"][::19] = 0
    T = synth.se3_exp(np.array([0.004, -0.003, 0.002, 0.001, -0.002, 0.0015]))
    r = reference.ref_sparse_residuals(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], p["cam"], p["T_ref_w"],
                                       synth.se3_mul(T, p["T_ref_w"]), p["px"], p["f"], p["pos"], p["has_point"], level)
    o = oracle.sparse_residuals(p["ref_pyr"][level], p["cur_pyr"][level], level, p["cam"], T, p["px"], p["f"], p["pos"],
                                p["has_point"], p["ref_pos"])
    v, m = o["visible"].astype(bool), o["in_image"].astype(bool)
    assert np.array_equal(r["visible"], o["visible"])
    assert r["visible_ref_patch_sha256"] == sha256(o["ref_patch"][v])
    assert r["n_meas"] == o["n_meas"] == 16 * int(m.sum()) and m.sum() > 200
    assert r["abs_res"].shape == (len(r["abs_res_rows"]), 16) and r["abs_res_rows"].max() < m.sum()
    # T_cur_from_ref is re-formed by the reference as T_cur_w * T_ref_w^-1 (1e-16 away from T): allow the rare pixel whose
    # f32 coordinate lands on the other side of a rounding boundary, demand identity for (nearly) all of them (of the
    # stored sample of in-image patches)
    res = np.abs(o["residuals"][m][r["abs_res_rows"]])
    same = res == r["abs_res"]
    assert same.mean() >= 0.99 and np.max(np.abs(res - r["abs_res"])) <= 1e-4
    assert abs(r["chi2"] - o["chi2"]) <= 1e-6 * abs(o["chi2"])
    assert np.allclose(r["H"], o["H"], rtol=1e-12, atol=1e-9 * np.abs(o["H"]).max())
    assert np.allclose(r["Jres"], o["Jres"], rtol=1e-9, atol=1e-6)


@pytest.mark.parametrize("seed", range(8))
def test_oracle_residual_pass_random_poses_equal_reference(oracle, seed, reference):
    """Randomised version of the residual pin: random scene seed, level, pose perturbation (up to 4 cm / 1 degree) and
    missing points; every quantity computeResiduals leaves behind must match (counts and patch cache exactly, per-pixel
    residual magnitudes bit for bit but for the rare coordinate on a rounding boundary)."""
    rng = np.random.default_rng(1000 + seed)
    p = synth.make_frame_pair(300 + seed, n_feat=int(rng.integers(40, 301)), n_levels=5)
    p["has_point"][rng.uniform(size=len(p["has_point"])) < 0.1] = 0
    level = int(rng.integers(0, 5))
    T = synth.se3_exp(np.concatenate([rng.uniform(-0.04, 0.04, 3), np.deg2rad(rng.uniform(-1.0, 1.0, 3))]))
    r = reference.ref_sparse_residuals(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], p["cam"], p["T_ref_w"],
                                       synth.se3_mul(T, p["T_ref_w"]), p["px"], p["f"], p["pos"], p["has_point"], level)
    o = oracle.sparse_residuals(p["ref_pyr"][level], p["cur_pyr"][level], level, p["cam"], T, p["px"], p["f"], p["pos"],
                                p["has_point"], p["ref_pos"])
    v, m = o["visible"].astype(bool), o["in_image"].astype(bool)
    assert np.array_equal(r["visible"], o["visible"]) and r["visible_ref_patch_sha256"] == sha256(o["ref_patch"][v])
    assert r["n_meas"] == o["n_meas"] == 16 * int(m.sum()) and m.sum() > 0
    d = np.abs(np.abs(o["residuals"][m][r["abs_res_rows"]]) - r["abs_res"])  # the stored sample of in-image patches
    assert (d == 0).mean() >= 0.99 and d.max() <= 1e-4
    assert abs(r["chi2"] - o["chi2"]) <= 1e-6 * abs(o["chi2"])
    assert np.allclose(r["H"], o["H"], rtol=1e-12, atol=1e-9 * np.abs(o["H"]).max())


@pytest.mark.parametrize("level", [0, 2, 4])
def test_oracle_residual_pass_with_patches_outside_the_image_equals_reference(oracle, level, reference):
    """computeResiduals' per-patch border test (sparse_img_align.cpp:190): features right up to the image border and a large
    motion, so that visible patches project outside the current image and are skipped -- the reference's n_meas_, the
    per-pixel |res| of the patches that stay, chi2, H_ and Jres_ vs the oracle."""
    rng = np.random.default_rng(5)
    cam = synth.camera_for(640, 480)
    plane, tex = synth.Plane.tilted(), synth.make_texture(7)
    T_ref_w = synth.base_pose()
    xi = np.array([0.07, -0.06, 0.05, np.deg2rad(1.2), np.deg2rad(-1.4), np.deg2rad(1.0)])
    T = synth.se3_exp(xi)
    ref_pyr = synth.build_pyramid(synth.render(cam, T_ref_w, plane, tex), 5)
    cur_pyr = synth.build_pyramid(synth.render(cam, synth.se3_mul(T, T_ref_w), plane, tex), 5)
    px = synth.jittered_features(rng, cam, 300, margin=4.0)
    f = cam.cam2world(px)
    pos = synth.intersect(plane, T_ref_w, f)
    hp = (rng.uniform(size=300) > 0.05).astype(np.uint8)
    ref_pos = synth.se3_inv(T_ref_w)[:, 3].copy()
    r = reference.ref_sparse_residuals(ref_pyr[0], cur_pyr[0], 5, cam, T_ref_w, synth.se3_mul(T, T_ref_w), px, f, pos, hp, level)
    o = oracle.sparse_residuals(ref_pyr[level], cur_pyr[level], level, cam, T, px, f, pos, hp, ref_pos)
    v, m = o["visible"].astype(bool), o["in_image"].astype(bool)
    assert np.array_equal(r["visible"], o["visible"])
    assert 0 < m.sum() < v.sum()  # the case really has visible patches that leave the current image
    assert r["n_meas"] == o["n_meas"] == 16 * int(m.sum())
    assert r["visible_ref_patch_sha256"] == sha256(o["ref_patch"][v])
    res = np.abs(o["residuals"][m][r["abs_res_rows"]])  # the stored sample of in-image patches
    same = res == r["abs_res"]
    assert same.mean() >= 0.99 and np.max(np.abs(res - r["abs_res"])) <= 1e-4
    assert abs(r["chi2"] - o["chi2"]) <= 1e-6 * abs(o["chi2"])
    assert np.allclose(r["H"], o["H"], rtol=1e-12, atol=1e-9 * np.abs(o["H"]).max())
    assert np.allclose(r["Jres"], o["Jres"], rtol=1e-9, atol=1e-5)


@pytest.mark.parametrize("n,outliers,noise,n_iter", [(8, 0.0, 0.5, 10), (40, 0.3, 1.0, 10), (1000, 0.1, 2.0, 3), (250, 0.03, 1.0, 1)])
def test_oracle_pose_optimizer_edge_cases_equal_reference_source_compiled_here(oracle, n, outliers, noise, n_iter, reference):
    """pose_optimizer::optimizeGaussNewton of the compiled reference at the corners of its behaviour: a handful of
    observations, a third of them gross outliers (Tukey weights, the culling of :129-145), few iterations (no convergence,
    the fixed scale of iteration 5 never reached)."""
    c = synth.make_pose_opt_case(90 + n, n=n, width=752, height=480, px_noise=noise, outlier_frac=outliers)
    r = reference.ref_pose_optimize(2.0, n_iter, c["cam"], c["T_init"], c["f"], c["pos"], c["level"], c["has_point"])
    o = oracle.pose_optimize(2.0, n_iter, c["cam"].fx, c["T_init"], c["f"], c["pos"], c["level"], c["has_point"])
    assert np.array_equal(r["has_point"], o["has_point"])
    assert r["num_obs"] == o["num_obs"]
    assert np.allclose(r["T"], o["T"], rtol=0, atol=1e-10)
    for k in ("estimated_scale", "error_init", "error_final"):
        assert np.isclose(r[k], o[k], rtol=1e-9), k


def test_oracle_pose_optimizer_equals_reference_source_compiled_here(oracle, reference):
    for seed in (3, 4):
        c = synth.make_pose_opt_case(seed, n=400)
        r = reference.ref_pose_optimize(2.0, 10, c["cam"], c["T_init"], c["f"], c["pos"], c["level"], c["has_point"])
        o = oracle.pose_optimize(2.0, 10, c["cam"].fx, c["T_init"], c["f"], c["pos"], c["level"], c["has_point"])
        assert np.array_equal(r["has_point"], o["has_point"])
        assert r["num_obs"] == o["num_obs"]
        assert np.allclose(r["T"], o["T"], rtol=0, atol=1e-10)
        for k in ("estimated_scale", "error_init", "error_final"):
            assert np.isclose(r[k], o[k], rtol=1e-9), k
        assert np.allclose(r["cov"], o["cov"], rtol=1e-6, atol=1e-12)


def test_oracle_point_optimize_equals_reference_source_compiled_here(oracle, reference):
    rng = np.random.default_rng(5)
    for _ in range(20):
        pos = np.array([rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(3, 6)])
        Ts, fs = [], []
        for _ in range(int(rng.integers(2, 7))):
            T = synth.se3_exp(np.concatenate([rng.uniform(-0.5, 0.5, 3), rng.uniform(-0.05, 0.05, 3)]))
            pc = T[:, :3] @ pos + T[:, 3]
            f = pc / np.linalg.norm(pc) + rng.normal(0, 1e-3, 3)
            Ts.append(T.reshape(12)); fs.append(f / np.linalg.norm(f))
        start = pos + rng.normal(0, 0.05, 3)
        for n_iter, tol in ((1, 1e-13), (3, 1e-13), (5, 1e-8)):
            # at convergence "new_chi2 > chi2" (point.cpp:152) compares rounding noise, so the roll-back of the last
            # ~1e-9 step can differ between two compilations of the same source; before that the runs agree to the ulp
            a = reference.ref_point_optimize(n_iter, start, np.array(Ts), np.array(fs))
            b = oracle.point_optimize(n_iter, start, np.array(Ts), np.array(fs))
            assert np.allclose(a, b, rtol=0, atol=tol), (n_iter, a - b)


def test_oracle_matcher_equals_reference_source_compiled_here(oracle, reference):
    """svo::Matcher::findMatchDirect (matcher.cpp:142-186: warp matrix, search level, warped patch, align1D/2D) of the
    compiled reference vs the oracle."""
    c = synth.make_match_case(21, 120)
    T_cur_ref = synth.se3_mul(c["T_cur_w"], synth.se3_inv(c["T_ref_w"]))
    ref_pos = synth.se3_inv(c["T_ref_w"])[:, 3]
    n_ok = 0
    for i in range(c["M"]):
        r = reference.ref_matcher(0, c["ref_pyr"][0], c["cur_pyr"][0], c["n_levels"], c["cam"], c["T_ref_w"], c["T_cur_w"],
                                  c["ref_px"][i], c["ref_f"][i], int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i],
                                  c["point_pos"][i], px_cur=c["px_cur"][i], n_pyr_levels=3)
        depth = np.linalg.norm(c["point_pos"][i] - ref_pos)
        o = oracle.find_match_direct(c["ref_pyr"], c["cur_pyr"], c["cam"], T_cur_ref, c["ref_px"][i], c["ref_f"][i],
                                     int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i], depth, 2, 10,
                                     c["px_cur"][i])
        assert r["success"] == o["success"], i
        assert r["search_level"] == o["search_level"], i
        assert np.allclose(r["A_cur_ref"], o["A_cur_ref"], rtol=1e-9, atol=1e-12), i
        if r["success"]:
            n_ok += 1
            assert np.allclose(r["px_cur"], o["px_cur"], rtol=0, atol=1e-9), i
    assert n_ok > c["M"] // 2


def test_oracle_epipolar_matcher_equals_reference_source_compiled_here(oracle, reference):
    """svo::Matcher::findEpipolarMatchDirect (matcher.cpp:188-330) of the compiled reference vs the oracle."""
    c = synth.make_depth_case(22, n_seeds=150)
    T_cur_ref = synth.se3_mul(c["T_cur_w"], synth.se3_inv(c["T_ref_w"]))
    n_ok = 0
    for i in range(c["M"]):
        mu, sig = 0.5, np.sqrt(float(c["seeds"]["sigma2"][i]))
        d_est, d_min, d_max = 1.0 / mu, 1.0 / (mu + sig), 1.0 / max(mu - sig, 1e-7)
        pos = synth.se3_inv(c["T_ref_w"])[:, :3] @ (c["ftr_f"][i] * d_est) + synth.se3_inv(c["T_ref_w"])[:, 3]
        r = reference.ref_matcher(1, c["ref_pyr"][0], c["cur_pyr"][0], c["n_levels"], c["cam"], c["T_ref_w"], c["T_cur_w"],
                                  c["ftr_px"][i], c["ftr_f"][i], int(c["ftr_level"][i]), int(c["ftr_type"][i]), c["ftr_grad"][i],
                                  pos, d_est=d_est, d_min=d_min, d_max=d_max, n_pyr_levels=3)
        o = oracle.find_epipolar_match_direct(c["ref_pyr"], c["cur_pyr"], c["cam"], T_cur_ref, c["ftr_px"][i], c["ftr_f"][i],
                                              int(c["ftr_level"][i]), int(c["ftr_type"][i]), c["ftr_grad"][i], d_est, d_min,
                                              d_max, 2)
        assert r["success"] == o["success"], i
        assert r["reject"] == o["reject"], i
        if r["success"]:
            n_ok += 1
            assert r["search_level"] == o["search_level"], i
            assert np.allclose(r["px_cur"], o["px_cur"], rtol=0, atol=1e-9), i
            assert np.isclose(r["depth"], o["depth"], rtol=1e-9), i
            assert np.isclose(r["epi_length"], o["epi_length"], rtol=1e-9), i
    assert n_ok > c["M"] // 4


def test_oracle_update_seed_equals_reference_source_compiled_here(oracle, reference):
    """DepthFilter::updateSeed / computeTau (depth_filter.cpp:309-357) as GCC compiles the reference source (default
    -ffp-contract=fast with FMA) vs the oracle's explicit-fma restatement: every f32 field bit for bit."""
    rng = np.random.default_rng(9)
    for _ in range(3000):
        a, b = np.float32(rng.uniform(1, 40)), np.float32(rng.uniform(1, 40))
        mu, zr = np.float32(rng.uniform(0.05, 2.0)), np.float32(rng.uniform(0.5, 4.0))
        s2 = np.float32(rng.uniform(1e-5, 1.0))
        x, tau2 = np.float32(mu + rng.normal(0, 0.3)), np.float32(10 ** rng.uniform(-7, -1))
        r = reference.ref_update_seed(x, tau2, a, b, mu, zr, s2)
        o = oracle.update_seed(x, tau2, a, b, mu, zr, s2)
        assert np.array_equal(r.view(np.uint32), o.view(np.uint32)), (r, o)
    for _ in range(500):
        T = synth.se3_exp(np.concatenate([rng.uniform(-0.5, 0.5, 3), rng.uniform(-0.1, 0.1, 3)]))
        f = rng.normal(size=3) * [0.3, 0.3, 0] + [0, 0, 1]
        f /= np.linalg.norm(f)
        z = rng.uniform(0.5, 10)
        # norms / dot products run inside the (stand-in) Eigen, whose summation order is [EXT]: equal to rounding
        assert np.isclose(reference.ref_compute_tau(T, f, z, 0.002), oracle.compute_tau(T, f, z, 0.002), rtol=1e-10, atol=0)


def test_oracle_depth_filter_equals_reference_source_compiled_here(oracle, reference):
    """svo::DepthFilter::updateSeeds of the compiled reference (depth_filter.cpp + matcher.cpp + feature_alignment.cpp)
    vs the oracle: same erase/converge/keep decision per seed and the same seed state bit for bit."""
    c = synth.make_depth_case(31, n_seeds=400)
    c["seeds"]["sigma2"][::5] *= np.float32(1e-3)   # some seeds close to convergence
    c["seeds"]["mu"][::5] = (1.0 / c["depth_gt"][::5]).astype(np.float32)
    r = reference.ref_depth_filter_update([c["ref_pyr"][0]], [c["T_ref_w"]], c["cur_pyr"][0], c["T_cur_w"], c["n_levels"], c["cam"],
                                          c["ref_index"], c["ftr_px"], c["ftr_f"], c["ftr_level"], c["ftr_type"], c["ftr_grad"],
                                          c["batch_id"], c["batch_counter"], c["seeds"])
    o = oracle.depth_filter_update([c["ref_pyr"]], [c["T_ref_w"]], c["cur_pyr"], c["T_cur_w"], c["cam"], c["ref_index"],
                                   c["ftr_px"], c["ftr_f"], c["ftr_level"], c["ftr_type"], c["ftr_grad"], c["batch_id"],
                                   c["batch_counter"], c["seeds"])
    st = o["status"]
    expect = np.where(st == 6, 1, np.where((st == 1) | (st == 7), 2, 0))
    assert np.array_equal(r["status"], expect)
    assert (st == 6).sum() > 5 and (st == 5).sum() > 50 and (st == 4).sum() > 0 and (st == 1).sum() > 0
    keep = expect == 0
    for k in ("a", "b", "mu", "z_range", "sigma2"):
        assert np.array_equal(r[k][keep].view(np.uint32), o[k][keep].view(np.uint32)), k
    conv = expect == 1
    assert np.array_equal(r["sigma2"][conv].view(np.uint32), o["sigma2"][conv].view(np.uint32))
    Tinv = synth.se3_inv(c["T_ref_w"])
    xyz = (c["ftr_f"][conv] / o["mu"][conv][:, None].astype(np.float64)) @ Tinv[:, :3].T + Tinv[:, 3]
    assert np.allclose(r["xyz_world"][conv], xyz, rtol=1e-12, atol=1e-12)


def _same_reprojection(a, b, px_tol=0.0):
    for k in ("n_matches", "n_trials", "n_new", "n_overlap"):
        assert a[k] == b[k], k
    for k in ("overlap_kf", "overlap_count", "new_point", "new_level", "new_type", "pt_type", "pt_n_failed", "pt_n_succeeded"):
        assert np.array_equal(a[k], b[k]), k
    assert np.max(np.abs(a["new_px"] - b["new_px"]), initial=0.0) <= px_tol
    assert np.allclose(a["new_grad"], b["new_grad"], rtol=0, atol=1e-9)


@pytest.mark.parametrize("seed,kw", [(5, {}), (6, dict(n_kfs=12, n_points=900)), (7, dict(bad_frac=0.5)),
                                     (8, dict(n_kfs=3, n_points=150, n_candidates=20))])
def test_oracle_reprojector_equals_reference_source_compiled_here(oracle, seed, kw, reference):
    """Reprojector::reprojectMap of the compiled reference (reprojector.cpp + map.cpp + matcher.cpp, real svo::Map /
    Frame / Feature / Point objects rebuilt from the flat view) vs the oracle's restatement: same overlap keyframes, same
    features added to the frame in the same order with identical pixels, same point counters / types / deletions."""
    c = synth.make_map_case(seed, **kw)
    o, r = oracle.reproject_map(c), reference.ref_reproject_map(c)
    _same_reprojection(o, r)
    # the reference cannot tell "erased while projecting" from "deleteCandidatePoint": both end in the candidates' trash
    assert np.array_equal(np.minimum(o["pt_action"], 2), np.minimum(r["pt_action"], 2))
    if not kw.get("n_kfs", 8) == 3:
        assert o["n_matches"] > 60 and o["n_trials"] > o["n_matches"]


def test_oracle_fast_detector_equals_reference_source_compiled_here(oracle, reference):
    """FastDetector::detect of the compiled reference (feature_detection.cpp; the un-vendored `fast` library and
    vk::shiTomasiScore restated once in oracle/fast_ext.h and linked behind both) vs the oracle's restatement of the grid
    logic: per-level scale, occupancy, strict best-score-per-cell, threshold."""
    for seed in (3, 4):
        d = synth.make_two_view(seed, n_levels=5)
        occ = (np.random.default_rng(seed).uniform(size=26 * 16) < 0.3).astype(np.uint8)
        for o_ in (None, occ):
            for thr in (20.0, 200.0):
                a = oracle.fast_detect(d["ref_pyr"], 3, 30, thr, o_)
                b = reference.ref_fast_detect(d["ref_pyr"][0], 5, 3, 30, thr, o_)
                assert all(np.array_equal(a[k], b[k]) for k in ("x", "y", "level"))
        assert len(a["x"]) > 20


def test_fast_ext_segment_test_properties(oracle):
    """Known answers of the [EXT] FAST restatement: a bright 3x3 blob corner on a dark background is a corner with score
    = contrast-1; straight edges and flat regions are not; detections keep a 3-pixel border."""
    img = np.full((40, 40), 50, np.uint8)
    img[20:, 20:] = 200                                                      # one L-corner at (20, 20)
    r = oracle.fast_detect([img], 1, 40, 0.0)
    assert len(r["x"]) == 1 and abs(int(r["x"][0]) - 20) <= 2 and abs(int(r["y"][0]) - 20) <= 2
    edge = np.full((40, 40), 50, np.uint8)
    edge[:, 20:] = 200                                                       # a straight edge: no FAST-10 corner
    assert len(oracle.fast_detect([edge], 1, 40, 0.0)["x"]) == 0
    assert len(oracle.fast_detect([np.full((40, 40), 9, np.uint8)], 1, 40, 0.0)["x"]) == 0


@pytest.mark.parametrize("seed,trans,rot", [(51, 0.12, 2.5), (52, 0.2, 4.0)])
def test_oracle_sia_large_motion_equals_reference_source_compiled_here(oracle, seed, trans, rot, reference):
    """Large inter-frame motion: patches leave the current image at the fine levels (the H of a pass then sums only the
    patches that contributed), levels end on rejected iterations, visibility flags stay set -- all reference behaviours
    the compiled reference and the oracle must share."""
    p = synth.make_frame_pair(seed, n_feat=250, trans=trans, rot_deg=rot)
    r = reference.ref_sparse_img_align(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], p["cam"], p["T_ref_w"], p["T_ref_w"],
                                       p["px"], p["f"], p["pos"], p["has_point"], 4, 0)
    o = oracle.sparse_img_align(p["ref_pyr"], p["cur_pyr"], p["cam"], synth.se3_identity(), p["px"], p["f"], p["pos"],
                                p["has_point"], p["ref_pos"], 4, 0)
    assert r["n_tracked"] == o["n_tracked"] and np.array_equal(r["visible"], o["visible"])
    assert np.allclose(r["T_cur_w"], synth.se3_mul(o["T"], p["T_ref_w"]), rtol=0, atol=1e-8)
    assert np.allclose(r["H"], o["H"], rtol=1e-8, atol=1e-8)
    n_vis = int(o["visible"].sum())
    assert any(t["n_meas"] // 16 < n_vis for t in o["trace"])               # some pass really lost patches


def test_oracle_depth_filter_two_keyframes_equals_reference_source_compiled_here(oracle, reference):
    """Seeds of two different keyframes updated by one frame (ref_index per seed), wide baseline, many edgelets."""
    a = synth.make_depth_case(61, n_seeds=300, baseline=0.5)
    b = synth.make_two_view(62, baseline=0.25)
    rng = np.random.default_rng(3)
    ref_index = rng.integers(0, 2, a["M"]).astype(np.int32)
    ftr_type = (rng.uniform(size=a["M"]) < 0.5).astype(np.int32)
    # keyframe 1 = the reference frame of a second two-view set rendered from the same plane; seeds keep their pixels
    kf_pyr, kf_T = [a["ref_pyr"], b["ref_pyr"]], [a["T_ref_w"], b["T_ref_w"]]
    r = reference.ref_depth_filter_update([k[0] for k in kf_pyr], kf_T, a["cur_pyr"][0], a["T_cur_w"], a["n_levels"], a["cam"],
                                          ref_index, a["ftr_px"], a["ftr_f"], a["ftr_level"], ftr_type, a["ftr_grad"], a["batch_id"],
                                          a["batch_counter"], a["seeds"])
    o = oracle.depth_filter_update(kf_pyr, kf_T, a["cur_pyr"], a["T_cur_w"], a["cam"], ref_index, a["ftr_px"], a["ftr_f"],
                                   a["ftr_level"], ftr_type, a["ftr_grad"], a["batch_id"], a["batch_counter"], a["seeds"])
    st = o["status"]
    assert np.array_equal(r["status"], np.where(st == 6, 1, np.where((st == 1) | (st == 7), 2, 0)))
    keep = r["status"] == 0
    for k in ("a", "b", "mu", "z_range", "sigma2"):
        assert np.array_equal(r[k][keep].view(np.uint32), o[k][keep].view(np.uint32)), k
    assert (st >= 5).sum() > 50


def test_oracle_matcher_wide_baseline_equals_reference_source_compiled_here(oracle, reference):
    """findMatchDirect under a strong affine warp (wide baseline, rotation about the optical axis): the search level leaves
    0 and the 10x10 warped patch samples the reference image far from the feature."""
    c = synth.make_match_case(71, 100, baseline=0.9, rot_deg=12.0)
    T_cur_ref = synth.se3_mul(c["T_cur_w"], synth.se3_inv(c["T_ref_w"]))
    ref_pos = synth.se3_inv(c["T_ref_w"])[:, 3]
    levels = []
    for i in range(c["M"]):
        r = reference.ref_matcher(0, c["ref_pyr"][0], c["cur_pyr"][0], c["n_levels"], c["cam"], c["T_ref_w"], c["T_cur_w"],
                                  c["ref_px"][i], c["ref_f"][i], int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i],
                                  c["point_pos"][i], px_cur=c["px_cur"][i], n_pyr_levels=3)
        o = oracle.find_match_direct(c["ref_pyr"], c["cur_pyr"], c["cam"], T_cur_ref, c["ref_px"][i], c["ref_f"][i],
                                     int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i],
                                     np.linalg.norm(c["point_pos"][i] - ref_pos), 2, 10, c["px_cur"][i])
        assert r["success"] == o["success"] and r["search_level"] == o["search_level"], i
        assert np.allclose(r["A_cur_ref"], o["A_cur_ref"], rtol=1e-9, atol=1e-12), i
        if r["success"]:
            assert np.allclose(r["px_cur"], o["px_cur"], rtol=0, atol=1e-9), i
        levels.append(o["search_level"])
    assert len(set(levels)) > 1


# ---- vk::halfSample / createImgPyramid: the rounding rule the reference's x86 build applies -------------------------------
@pytest.mark.parametrize("size,levels", [((640, 480), 5), ((752, 480), 5), ((1920, 1080), 6), ((656, 490), 5), ((70, 50), 3)])
def test_pyramid_rule_reference_source_compiled_here(oracle, size, levels, reference):
    """oracle/_ref = the reference's own frame.cpp (createImgPyramid) over the restated vk::halfSample with REAL SSE2
    intrinsics (the branch vikit takes when cols % 16 == 0 and the buffers are 16-byte aligned).  The oracle's plain-C
    restatement of that rule (PYR_X86) and the numpy one must equal it bit for bit at every level; the scalar rule must
    NOT wherever the SSE2 branch is taken."""
    from rpg_svo_b200 import synth

    w, h = size
    img = np.random.default_rng(w + 3 * h).integers(0, 256, (h, w), dtype=np.uint8)
    ref = reference.ref_image_pyramid(img, levels)
    cur = img
    for l in range(levels):
        assert ref[l] == sha256(cur), f"level {l}"  # the reference's levels are stored as SHA-256 digests
        if l + 1 < levels:
            nxt = oracle.half_sample(cur, oracle.PYR_X86)
            assert np.array_equal(nxt, synth.half_sample(cur, synth.PYR_X86))
            if cur.shape[1] % 16 == 0:
                assert not np.array_equal(nxt, oracle.half_sample(cur, oracle.PYR_SCALAR))
            cur = nxt
