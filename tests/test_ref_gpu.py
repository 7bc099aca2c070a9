"""GPU parity against oracle/_ref: the reference's OWN classes (svo::SparseImgAlign, svo::pose_optimizer,
svo::DepthFilter with svo::Matcher and svo::feature_alignment) compiled from the reference's svo/src against stand-in
third-party headers (oracle/shim), their outputs on these inputs stored under tests/golden/reference/.  These tests call
the CUDA path through the C ABI and compare with the reference's outputs directly -- no oracle restatement in between."""
import numpy as np
import pytest

from rpg_svo_b200 import synth
from tests.reference_outputs import sha256

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed,levels", [(41, (4, 2)), (42, (4, 0))])
def test_sparse_img_align_vs_compiled_reference(ctx, reference, seed, levels):
    p = synth.make_frame_pair(seed, n_feat=300)
    p["has_point"][::23] = 0
    r = reference.ref_sparse_img_align(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], p["cam"], p["T_ref_w"], p["T_ref_w"],
                                       p["px"], p["f"], p["pos"], p["has_point"], levels[0], levels[1])
    fr, fc = ctx.frame(p["ref_pyr"]), ctx.frame(p["cur_pyr"])
    g = ctx.sparse_img_align(fr, fc, p["cam"], synth.se3_identity(), p["px"], p["f"], p["pos"], p["has_point"],
                             p["ref_pos"], levels[0], levels[1], 30, want_trace=False)
    fr.destroy(); fc.destroy()
    assert g["n_tracked"] == r["n_tracked"]
    assert np.array_equal(g["visible"], r["visible"])                     # bit-exact mask
    dt, dr = synth.pose_error(synth.se3_mul(g["T"], p["T_ref_w"]), r["T_cur_w"])
    assert dt <= 1e-4 and dr <= 1e-4, (dt, dr)                            # north_star tolerance on the final SE3
    assert synth.pose_error(r["T_cur_w"], p["T_cur_w"])[0] < 1e-3         # and the reference really tracked the motion


@pytest.mark.parametrize("level", [0, 2, 4])
def test_residual_pass_vs_compiled_reference(ctx, reference, level):
    """The kernel's residual pass against the reference's own computeResiduals object code (no oracle in between): masks
    and patch cache bit-exact, every per-pixel residual magnitude within the north_star's 1e-4 (and bit-identical for
    nearly all pixels), chi2 / n_meas / Jres_ / H_."""
    p = synth.make_frame_pair(45, n_feat=300, n_levels=5)
    p["has_point"][::19] = 0
    T = synth.se3_exp(np.array([0.004, -0.003, 0.002, 0.001, -0.002, 0.0015]))
    r = reference.ref_sparse_residuals(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], p["cam"], p["T_ref_w"],
                                       synth.se3_mul(T, p["T_ref_w"]), p["px"], p["f"], p["pos"], p["has_point"], level)
    fr, fc = ctx.frame(p["ref_pyr"]), ctx.frame(p["cur_pyr"])
    g = ctx.sparse_residuals(fr, fc, p["cam"], level, T, p["px"], p["f"], p["pos"], p["has_point"], p["ref_pos"])
    fr.destroy(); fc.destroy()
    v, m = g["visible"].astype(bool), g["in_image"].astype(bool)
    assert np.array_equal(g["visible"], r["visible"])
    assert sha256(g["ref_patch"][v]) == r["visible_ref_patch_sha256"]
    assert g["n_meas"] == r["n_meas"] == 16 * int(m.sum()) and m.sum() > 200
    d = np.abs(np.abs(g["residuals"][m][r["abs_res_rows"]]) - r["abs_res"])  # the stored sample of in-image patches
    assert d.max() <= 1e-4 and (d == 0).mean() >= 0.99, (d.max(), (d == 0).mean())
    assert abs(g["chi2"] - r["chi2"]) <= 1e-5 * abs(r["chi2"])
    assert np.allclose(g["H"], r["H"], rtol=1e-9, atol=1e-6)
    assert np.allclose(g["Jres"], r["Jres"], rtol=1e-5, atol=1e-3)


def test_pose_optimizer_vs_compiled_reference(ctx, reference):
    c = synth.make_pose_opt_case(43, 800, 752, 480)
    r = reference.ref_pose_optimize(2.0, 10, c["cam"], c["T_init"], c["f"], c["pos"], c["level"], c["has_point"])
    g = ctx.pose_optimize(2.0, 10, c["cam"].fx, c["T_init"], c["f"], c["pos"], c["level"], c["has_point"])
    assert np.array_equal(g["has_point"], r["has_point"]) and g["num_obs"] == r["num_obs"]
    dt, dr = synth.pose_error(g["T"], r["T"])
    assert dt < 1e-8 and dr < 1e-8
    for k in ("estimated_scale", "error_init", "error_final"):
        assert abs(g[k] - r[k]) <= 1e-9 * max(1.0, abs(r[k])), k
    assert np.allclose(g["cov"], r["cov"], rtol=1e-6, atol=1e-12)


def test_depth_filter_vs_compiled_reference(ctx, reference):
    c = synth.make_depth_case(44, n_seeds=1000)
    c["seeds"]["sigma2"][::5] *= np.float32(1e-3)
    c["seeds"]["mu"][::5] = (1.0 / c["depth_gt"][::5]).astype(np.float32)
    r = reference.ref_depth_filter_update([c["ref_pyr"][0]], [c["T_ref_w"]], c["cur_pyr"][0], c["T_cur_w"], c["n_levels"], c["cam"],
                                          c["ref_index"], c["ftr_px"], c["ftr_f"], c["ftr_level"], c["ftr_type"], c["ftr_grad"],
                                          c["batch_id"], c["batch_counter"], c["seeds"])
    fr, fc = ctx.frame(c["ref_pyr"]), ctx.frame(c["cur_pyr"])
    g = ctx.depth_filter_update([fr], [c["T_ref_w"]], fc, c["T_cur_w"], c["cam"], c["ref_index"], c["ftr_px"], c["ftr_f"],
                                c["ftr_level"], c["ftr_type"], c["ftr_grad"], c["batch_id"], c["batch_counter"], c["seeds"])
    fr.destroy(); fc.destroy()
    st = g["status"]
    assert np.array_equal(r["status"], np.where(st == 6, 1, np.where((st == 1) | (st == 7), 2, 0)))  # keep/converge/erase
    keep = r["status"] == 0
    nomatch = st == 4
    assert nomatch.sum() > 0 and np.array_equal(g["b"][nomatch], r["b"][nomatch])  # b++ on failed matches: exact
    for k in ("a", "b", "mu", "sigma2"):                                   # expf is the one non-bit-exact device op
        assert np.allclose(g[k][keep], r[k][keep], rtol=2e-5, atol=1e-7), k
    assert (st == 6).sum() > 10 and (st == 5).sum() > 200


def test_find_match_direct_vs_compiled_reference(ctx, reference):
    c = synth.make_match_case(45, 150)
    fr, fc = ctx.frame(c["ref_pyr"]), ctx.frame(c["cur_pyr"])
    g = ctx.find_match_direct([fr], [c["T_ref_w"]], fc, c["T_cur_w"], c["cam"], np.zeros(c["M"], np.int32), c["ref_px"],
                              c["ref_f"], c["ref_level"], c["ftr_type"], c["ref_grad"], c["point_pos"], c["px_cur"],
                              max_search_level=2)
    fr.destroy(); fc.destroy()
    n_ok = 0
    for i in range(c["M"]):
        r = reference.ref_matcher(0, c["ref_pyr"][0], c["cur_pyr"][0], c["n_levels"], c["cam"], c["T_ref_w"], c["T_cur_w"],
                                  c["ref_px"][i], c["ref_f"][i], int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i],
                                  c["point_pos"][i], px_cur=c["px_cur"][i], n_pyr_levels=3)
        assert bool(g["success"][i]) == r["success"], i
        assert g["search_level"][i] == r["search_level"], i
        if r["success"]:
            n_ok += 1
            assert np.max(np.abs(g["px_cur"][i] - r["px_cur"])) <= 1e-4, i
    assert n_ok > c["M"] // 2
