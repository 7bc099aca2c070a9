"""GPU parity of svo_b200_fast_detect ("next" row f4: feature_detection::FastDetector::detect,
svo/src/feature_detection.cpp:66-115) against the oracle and against the reference's own FastDetector object code
(oracle/_ref; the un-vendored `fast` library and vk::shiTomasiScore are restated in oracle/fast_ext.h in both)."""
import numpy as np
import pytest

from rpg_svo_b200 import synth

pytestmark = pytest.mark.gpu


def _same(g, o):
    for k in ("x", "y", "level"):
        assert np.array_equal(g[k], o[k]), k          # integer work: bit-exact
    if "score" in o:
        assert np.array_equal(g["score"].view(np.uint32), o["score"].view(np.uint32))  # same f32 bits


@pytest.mark.parametrize("size,seed", [((752, 480), 3), ((640, 480), 4), ((1920, 1080), 5), ((97, 61), 6)])
def test_fast_detect_matches_oracle(ctx, oracle, size, seed):
    d = synth.make_two_view(seed, width=size[0], height=size[1], n_levels=4)
    pyr = d["ref_pyr"]
    fr = ctx.frame(pyr)
    rng = np.random.default_rng(seed)
    n_cells = int(np.ceil(size[0] / 30)) * int(np.ceil(size[1] / 30))
    for occ in (None, (rng.uniform(size=n_cells) < 0.4).astype(np.uint8)):
        for thr in (20.0, 150.0):
            g = ctx.fast_detect(fr, 30, 3, thr, occ)
            o = oracle.fast_detect(pyr, 3, 30, thr, occ, cap=8192)
            _same(g, o)
            assert g["n"] == len(o["x"])
    fr.destroy()


def test_fast_detect_noise_image_and_options(ctx, oracle):
    """Dense corners everywhere (uniform noise) stress ties in the non-maximum suppression and the per-cell arg-max."""
    rng = np.random.default_rng(11)
    img = rng.integers(0, 256, (240, 320), dtype=np.uint8)
    img[100:140, 100:200] = 128                                              # a flat region: no corners
    pyr = synth.build_pyramid(img, 3)
    fr = ctx.frame(pyr)
    for cell, levels, ties in ((30, 3, 0), (16, 1, 1), (50, 2, 0), (30, 3, 1)):
        g = ctx.fast_detect(fr, cell, levels, 20.0, nonmax_ties_suppress=ties)
        o = oracle.fast_detect(pyr, levels, cell, 20.0, cap=8192, nonmax_ties_suppress=ties)
        _same(g, o)
    fr.destroy()


def test_fast_detect_vs_compiled_reference(ctx, oracle, reference):
    d = synth.make_two_view(7, n_levels=5)
    fr = ctx.frame(d["ref_pyr"])
    occ = (np.random.default_rng(2).uniform(size=26 * 16) < 0.3).astype(np.uint8)
    g = ctx.fast_detect(fr, 30, 3, 20.0, occ)
    r = reference.ref_fast_detect(d["ref_pyr"][0], 5, 3, 30, 20.0, occ)
    _same(g, r)
    assert len(r["x"]) > 100
    fr.destroy()


def test_fast_detect_flat_and_errors(ctx):
    from rpg_svo_b200.capi import SvoB200Error
    pyr = synth.build_pyramid(np.full((120, 160), 77, np.uint8), 3)
    fr = ctx.frame(pyr)
    g = ctx.fast_detect(fr, 30, 3, 20.0)
    assert g["n"] == 0
    with pytest.raises(SvoB200Error):
        ctx.fast_detect(fr, 30, 5, 20.0)                                     # more levels than the pyramid has
    with pytest.raises(SvoB200Error):
        ctx.fast_detect(fr, 0, 3, 20.0)
    fr.destroy()
