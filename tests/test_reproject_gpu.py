"""GPU parity of svo_b200_reproject_map ("next" row f2: Reprojector::reprojectMap, svo/src/reprojector.cpp:64-217):
speculative device alignment of every in-frame map point + host replay of the cell policy, against the sequential oracle
and against the reference's own Reprojector/Map object code (oracle/_ref)."""
import numpy as np
import pytest

from rpg_svo_b200 import synth

pytestmark = pytest.mark.gpu


def _run_gpu(ctx, c, **opt_over):
    kfs = [ctx.frame(p) for p in c["kf_pyr"]]
    cur = ctx.frame(c["cur_pyr"])
    opt = dict(c["options"], **opt_over)
    g = ctx.reproject_map(c["view"], kfs, cur, c["cur_T_f_w"], c["cam"], opt, c["cell_order"], c["pt_type"], c["pt_n_failed"],
                          c["pt_n_succeeded"])
    for f in kfs:
        f.destroy()
    cur.destroy()
    return g


def _same(g, o):
    for k in ("n_matches", "n_trials", "n_new", "n_overlap"):
        assert g[k] == o[k], k
    for k in ("overlap_kf", "overlap_count", "new_point", "new_level", "new_type", "pt_type", "pt_n_failed", "pt_n_succeeded"):
        assert np.array_equal(g[k], o[k]), k                                  # integer / index work: bit-exact
    assert np.max(np.abs(g["new_px"] - o["new_px"]), initial=0.0) <= 1e-4     # refined pixels
    assert np.allclose(g["new_grad"], o["new_grad"], rtol=0, atol=1e-9)


@pytest.mark.parametrize("seed,kw", [(5, {}), (6, dict(n_kfs=12, n_points=900)), (7, dict(bad_frac=0.5)),
                                     (8, dict(n_kfs=3, n_points=150, n_candidates=20))])
def test_reproject_map_matches_oracle(ctx, oracle, seed, kw):
    c = synth.make_map_case(seed, **kw)
    g, o = _run_gpu(ctx, c), oracle.reproject_map(c)
    _same(g, o)
    assert np.array_equal(g["pt_action"], o["pt_action"])
    assert g["n_projected"] == o["n_projected"]
    assert g["n_speculative"] >= g["n_trials"] - (c["pt_type"] == 0).sum()   # the device aligned more than the policy used


def test_reproject_map_vs_compiled_reference(ctx, oracle, reference):
    c = synth.make_map_case(9, n_kfs=10, n_points=800)
    g, r = _run_gpu(ctx, c), reference.ref_reproject_map(c)
    _same(g, r)
    assert np.array_equal(np.minimum(g["pt_action"], 2), np.minimum(r["pt_action"], 2))
    assert g["n_matches"] == c["options"]["max_fts"] + 1                     # the maxFts stop was reached


def test_reproject_map_policy_variants(ctx, oracle):
    c = synth.make_map_case(10)
    for over in (dict(max_fts=30), dict(max_n_kfs=2), dict(grid_size=60), dict(max_search_level=0)):
        cc = dict(c, options=dict(c["options"], **over))
        if "grid_size" in over:
            n_cells = int(np.ceil(c["cam"].width / 60)) * int(np.ceil(c["cam"].height / 60))
            cc["cell_order"] = np.random.default_rng(1).permutation(n_cells).astype(np.int32)
        g, o = _run_gpu(ctx, cc), oracle.reproject_map(cc)
        _same(g, o)


def test_reproject_map_empty_and_errors(ctx):
    from rpg_svo_b200.capi import SvoB200Error
    c = synth.make_map_case(11, n_kfs=3, n_points=60, n_candidates=5)
    v = dict(c["view"])
    v["kf_keypt_valid"] = np.zeros_like(v["kf_keypt_valid"])                 # no keyframe overlaps, no candidates
    v["n_candidates"] = 0
    g = _run_gpu(ctx, dict(c, view=v))
    assert g["n_matches"] == 0 and g["n_new"] == 0 and g["n_overlap"] == 0
    bad = dict(c["view"])
    bad["pt_obs"] = np.full_like(bad["pt_obs"], 10 ** 6)
    with pytest.raises(SvoB200Error):
        _run_gpu(ctx, dict(c, view=bad))
    with pytest.raises(SvoB200Error):
        _run_gpu(ctx, c, max_search_level=9)
