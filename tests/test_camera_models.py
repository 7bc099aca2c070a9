"""Distorted camera models ([EXT] vk::PinholeCamera with radial-tangential coefficients, vk::ATANCamera) with the
parameters the reference ships (svo_ros/param/camera_pinhole.yaml, camera_atan.yaml).

CPU: the oracle's restatement vs an independent numpy one and vs oracle/_ref (the reference's own SparseImgAlign /
Matcher running over the shim's restated vikit camera classes).  GPU: every kernel that calls the camera
(SparseImgAlign, findMatchDirect, DepthFilter::updateSeeds / findEpipolarMatchDirect, Reprojector) vs the oracle."""
import numpy as np
import pytest

from rpg_svo_b200 import synth

CAMERAS = ["atan", "pinhole_radtan"]


@pytest.mark.parametrize("kind", CAMERAS)
def test_camera_functions_oracle_vs_numpy(oracle, kind):
    cam = synth.reference_param_camera(kind)
    rng = np.random.default_rng(3)
    px = np.stack([rng.uniform(5, 746, 4000), rng.uniform(5, 474, 4000)], axis=1)
    f = oracle.camera_cam2world(cam, px)
    assert np.allclose(np.linalg.norm(f, axis=1), 1.0, atol=1e-15)
    assert np.allclose(f, cam.cam2world(px), rtol=0, atol=1e-12)
    xyz = f * rng.uniform(0.5, 5.0, (4000, 1))
    assert np.allclose(oracle.camera_world2cam(cam, xyz), cam.world2cam(xyz), rtol=0, atol=1e-9)
    back = oracle.camera_world2cam(cam, xyz)
    if kind == "atan":  # closed-form inverse: exact round trip
        assert np.max(np.abs(back - px)) < 1e-9
    else:  # vikit's cam2world = OpenCV's 5 fixed-point iterations on a float point: sub-pixel only, worst at the corners
        assert np.median(np.abs(back - px)) < 0.1 and np.max(np.abs(back - px)) < 1.0


@pytest.mark.parametrize("kind", CAMERAS)
def test_oracle_sparse_img_align_distorted_equals_reference_source_compiled_here(oracle, kind, reference):
    """The reference's SparseImgAlign (oracle/_ref) over the shim's vk::ATANCamera / distorted vk::PinholeCamera vs the
    oracle: same visibility, same pose."""
    cam = synth.reference_param_camera(kind)
    p = synth.make_frame_pair(61, n_feat=200, cam=cam)
    r = reference.ref_sparse_img_align(p["ref_pyr"][0], p["cur_pyr"][0], p["n_levels"], cam, p["T_ref_w"], p["T_ref_w"], p["px"],
                                       p["f"], p["pos"], p["has_point"], 4, 0)
    o = oracle.sparse_img_align(p["ref_pyr"], p["cur_pyr"], cam, synth.se3_identity(), p["px"], p["f"], p["pos"],
                                p["has_point"], p["ref_pos"], 4, 0)
    assert r["n_tracked"] == o["n_tracked"] > 100
    assert np.array_equal(r["visible"], o["visible"])
    assert np.allclose(r["T_cur_w"], synth.se3_mul(o["T"], p["T_ref_w"]), rtol=0, atol=1e-9)
    assert synth.pose_error(o["T"], p["T_cur_ref_gt"])[0] < 2e-3  # the distorted model really tracks the motion


@pytest.mark.parametrize("kind", CAMERAS)
def test_oracle_matcher_distorted_equals_reference_source_compiled_here(oracle, kind, reference):
    cam = synth.reference_param_camera(kind)
    c = synth.make_match_case(23, 60, cam=cam)
    T_cur_ref = synth.se3_mul(c["T_cur_w"], synth.se3_inv(c["T_ref_w"]))
    ref_pos = synth.se3_inv(c["T_ref_w"])[:, 3]
    n_ok = 0
    for i in range(c["M"]):
        r = reference.ref_matcher(0, c["ref_pyr"][0], c["cur_pyr"][0], c["n_levels"], cam, c["T_ref_w"], c["T_cur_w"],
                                  c["ref_px"][i], c["ref_f"][i], int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i],
                                  c["point_pos"][i], px_cur=c["px_cur"][i], n_pyr_levels=3)
        depth = np.linalg.norm(c["point_pos"][i] - ref_pos)
        o = oracle.find_match_direct(c["ref_pyr"], c["cur_pyr"], cam, T_cur_ref, c["ref_px"][i], c["ref_f"][i],
                                     int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i], depth, 2, 10, c["px_cur"][i])
        assert r["success"] == o["success"] and r["search_level"] == o["search_level"], i
        assert np.allclose(r["A_cur_ref"], o["A_cur_ref"], rtol=1e-9, atol=1e-12), i
        if r["success"]:
            n_ok += 1
            assert np.allclose(r["px_cur"], o["px_cur"], rtol=0, atol=1e-9), i
    assert n_ok > c["M"] // 2


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind", CAMERAS)
@pytest.mark.parametrize("geometry", [(-1, 0), (1, 1), (1, 2)])
def test_gpu_sparse_img_align_distorted(ctx, oracle, kind, geometry):
    cam = synth.reference_param_camera(kind)
    d = synth.make_frame_pair(62, n_feat=300, cam=cam)
    ctx.sia_config(*geometry)
    ref, cur = ctx.frame(d["ref_pyr"]), ctx.frame(d["cur_pyr"])
    g = ctx.sparse_img_align(ref, cur, cam, synth.se3_identity(), d["px"], d["f"], d["pos"], d["has_point"], d["ref_pos"], 4, 0,
                             want_trace=True)
    ctx.sia_config(-1, 0)
    o = oracle.sparse_img_align(d["ref_pyr"], d["cur_pyr"], cam, synth.se3_identity(), d["px"], d["f"], d["pos"], d["has_point"],
                                d["ref_pos"], 4, 0)
    dt, dr = synth.pose_error(g["T"], o["T"])
    assert dt <= 1e-4 and dr <= 1e-4, (dt, dr)
    assert np.array_equal(g["visible"], o["visible"]) and g["n_tracked"] == o["n_tracked"]
    assert [(t["level"], t["iter"], t["n_meas"]) for t in g["trace"]] == [(t["level"], t["iter"], t["n_meas"]) for t in o["trace"]]
    ref.destroy(); cur.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", CAMERAS)
def test_gpu_find_match_direct_distorted(ctx, oracle, kind):
    cam = synth.reference_param_camera(kind)
    c = synth.make_match_case(24, 200, cam=cam)
    ref, cur = ctx.frame(c["ref_pyr"]), ctx.frame(c["cur_pyr"])
    g = ctx.find_match_direct([ref], [c["T_ref_w"]], cur, c["T_cur_w"], cam, np.zeros(c["M"], np.int32), c["ref_px"], c["ref_f"],
                              c["ref_level"], c["ftr_type"], c["ref_grad"], c["point_pos"], c["px_cur"], 2)
    T_cur_ref = synth.se3_mul(c["T_cur_w"], synth.se3_inv(c["T_ref_w"]))
    ref_pos = synth.se3_inv(c["T_ref_w"])[:, 3]
    n_ok = 0
    for i in range(c["M"]):
        o = oracle.find_match_direct(c["ref_pyr"], c["cur_pyr"], cam, T_cur_ref, c["ref_px"][i], c["ref_f"][i],
                                     int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i],
                                     np.linalg.norm(c["point_pos"][i] - ref_pos), 2, 10, c["px_cur"][i])
        assert bool(g["success"][i]) == bool(o["success"]) and g["search_level"][i] == o["search_level"], i
        assert np.allclose(g["A_cur_ref"][i], o["A_cur_ref"], rtol=1e-7, atol=1e-9), i
        if o["success"]:
            n_ok += 1
            assert np.max(np.abs(g["px_cur"][i] - o["px_cur"])) <= 1e-4, i
    assert n_ok > c["M"] // 2
    ref.destroy(); cur.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", CAMERAS)
def test_gpu_depth_filter_distorted(ctx, oracle, kind):
    cam = synth.reference_param_camera(kind)
    c = synth.make_depth_case(25, 400, cam=cam)
    ref, cur = ctx.frame(c["ref_pyr"]), ctx.frame(c["cur_pyr"])
    args = (c["ref_index"], c["ftr_px"], c["ftr_f"], c["ftr_level"], c["ftr_type"], c["ftr_grad"], c["batch_id"], c["batch_counter"],
            c["seeds"])
    g = ctx.depth_filter_update([ref], [c["T_ref_w"]], cur, c["T_cur_w"], cam, *args)
    o = oracle.depth_filter_update([c["ref_pyr"]], [c["T_ref_w"]], c["cur_pyr"], c["T_cur_w"], cam, *args)
    assert np.array_equal(g["status"], o["status"]) and np.array_equal(g["n_zmssd"], o["n_zmssd"])
    upd = o["status"] >= 5
    assert upd.sum() > 0.25 * len(upd)
    assert np.max(np.abs(g["px_cur"][upd] - o["px_cur"][upd])) <= 1e-4
    assert np.allclose(g["z"][upd], o["z"][upd], rtol=1e-6)
    for k in ("a", "b", "mu", "sigma2"):
        assert np.allclose(g[k], o[k], rtol=2e-5, atol=1e-7), k
    ref.destroy(); cur.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", CAMERAS)
def test_gpu_reprojector_distorted(ctx, oracle, kind):
    cam = synth.reference_param_camera(kind)
    m = synth.make_map_case(26, n_kfs=6, n_points=500, n_candidates=60, cam=cam)
    kfs, cur = [ctx.frame(p) for p in m["kf_pyr"]], ctx.frame(m["cur_pyr"])
    g = ctx.reproject_map(m["view"], kfs, cur, m["cur_T_f_w"], cam, m["options"], m["cell_order"], m["pt_type"], m["pt_n_failed"],
                          m["pt_n_succeeded"])
    o = oracle.reproject_map(m)
    assert g["n_matches"] == o["n_matches"] > 20
    assert np.array_equal(g["new_point"], o["new_point"]) and np.array_equal(g["new_level"], o["new_level"])
    assert np.max(np.abs(g["new_px"] - o["new_px"])) <= 1e-4
    assert np.array_equal(g["pt_type"], o["pt_type"]) and np.array_equal(g["pt_n_failed"], o["pt_n_failed"])
    for f in kfs:
        f.destroy()
    cur.destroy()
