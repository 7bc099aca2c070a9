"""GPU parity: align2D / align1D / findMatchDirect kernels vs the CPU oracle (bit-exact: the kernels
replay the reference's float operations in the reference's order)."""
import numpy as np
import pytest

from rpg_svo_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def case():
    return synth.make_align_case(11, 400)


@pytest.mark.parametrize("n_iter", [3, 10])
def test_align2d_batch_bit_exact(ctx, oracle, case, n_iter):
    c = case
    fr = ctx.frame(c["pyr"])
    conv, px = ctx.align2d_batch(fr, c["level"], c["pwb"], c["patch"], n_iter, c["px_start"])
    n_conv = 0
    for i in range(len(c["level"])):
        ok, p = oracle.align2d(c["pyr"][c["level"][i]], c["pwb"][i], c["patch"][i], n_iter, c["px_start"][i])
        assert ok == conv[i], i
        assert np.array_equal(p, px[i]), (i, p, px[i])
        n_conv += ok
    assert n_conv > (0.9 if n_iter >= 10 else 0.2) * len(conv)  # the problems are well posed
    err = np.linalg.norm(px[conv] - c["px_true"][conv], axis=1)
    assert np.median(err) < 0.1  # sanity band of svo/test/test_feature_alignment.cpp:98 (0.015 px on real data)
    fr.destroy()


def test_align1d_batch_bit_exact(ctx, oracle, case):
    c = case
    fr = ctx.frame(c["pyr"])
    conv, px, h_inv = ctx.align1d_batch(fr, c["level"], c["dir"], c["pwb"], c["patch"], 10, c["px_start"])
    for i in range(len(c["level"])):
        ok, p, h = oracle.align1d(c["pyr"][c["level"][i]], c["dir"][i], c["pwb"][i], c["patch"][i], 10, c["px_start"][i])
        assert ok == conv[i], i
        assert np.array_equal(p, px[i]), (i, p, px[i])
        assert h == h_inv[i]
    fr.destroy()


def test_align_empty_batch(ctx, case):
    fr = ctx.frame(case["pyr"])
    conv, px = ctx.align2d_batch(fr, np.zeros(0, np.int32), np.zeros((0, 100), np.uint8), np.zeros((0, 64), np.uint8), 10,
                                 np.zeros((0, 2)))
    assert len(conv) == 0
    fr.destroy()


def test_find_match_direct(ctx, oracle):
    c = synth.make_match_case(21, 300)
    ref, cur = ctx.frame(c["ref_pyr"]), ctx.frame(c["cur_pyr"])
    g = ctx.find_match_direct([ref], [c["T_ref_w"]], cur, c["T_cur_w"], c["cam"], np.zeros(c["M"], np.int32),
                              c["ref_px"], c["ref_f"], c["ref_level"], c["ftr_type"], c["ref_grad"], c["point_pos"],
                              c["px_cur"], max_search_level=2)
    T_cur_ref = oracle.se3_mul(c["T_cur_w"], oracle.se3_inv(c["T_ref_w"]))
    ref_pos = oracle.se3_inv(c["T_ref_w"])[:, 3]
    n_ok = 0
    for i in range(c["M"]):
        depth = float(np.linalg.norm(ref_pos - c["point_pos"][i]))
        o = oracle.find_match_direct(c["ref_pyr"], c["cur_pyr"], c["cam"], T_cur_ref, c["ref_px"][i], c["ref_f"][i],
                                     int(c["ref_level"][i]), int(c["ftr_type"][i]), c["ref_grad"][i], depth, 2, 10,
                                     c["px_cur"][i])
        assert o["success"] == g["success"][i], i
        assert o["search_level"] == g["search_level"][i]
        assert np.allclose(o["A_cur_ref"], g["A_cur_ref"][i], rtol=1e-9, atol=1e-12)
        assert np.max(np.abs(o["px_cur"] - g["px_cur"][i])) <= 1e-4, (i, o["px_cur"], g["px_cur"][i])
        n_ok += o["success"]
    assert n_ok > 0.5 * c["M"]
    ok = g["success"]
    assert np.median(np.linalg.norm(g["px_cur"][ok] - c["px_cur_true"][ok], axis=1)) < 0.3
    ref.destroy(); cur.destroy()


def test_align_kernels_equal_reference_source_compiled(ctx, oracle, case, reference):
    """GPU kernels vs oracle/_ref (the reference's own feature_alignment.cpp compiled with stand-in headers):
    bit-identical pixel estimates and convergence flags."""
    c = case
    fr = ctx.frame(c["pyr"])
    conv, px = ctx.align2d_batch(fr, c["level"], c["pwb"], c["patch"], 10, c["px_start"])
    conv1, px1, h1 = ctx.align1d_batch(fr, c["level"], c["dir"], c["pwb"], c["patch"], 10, c["px_start"])
    for i in range(len(c["level"])):
        img = c["pyr"][c["level"][i]]
        ok, p = reference.ref_align2d(img, c["pwb"][i], c["patch"][i], 10, c["px_start"][i])
        assert ok == conv[i] and np.array_equal(p, px[i]), i
        ok, p, h = reference.ref_align1d(img, c["dir"][i], c["pwb"][i], c["patch"][i], 10, c["px_start"][i])
        assert ok == conv1[i] and np.array_equal(p, px1[i]) and h == h1[i], i
    fr.destroy()
