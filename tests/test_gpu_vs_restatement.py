"""The CUDA path against stored restatement outputs, on any B200.

tests/golden/restatement_outputs.npz holds what the CPU oracle and tests/assoc_ref.py compute on the seeded inputs of
tests/restated_cases.py, the same inputs tests/test_gpu_vs_reference.py runs through the reference's own compiled code
where oracle/_ref is built. tests/test_reference_pin.py checks the stored values against that code wherever it is present.
Arrays stored only as probes are also compared element by element with the restatement run here. Tolerances as in
tests/test_gpu_vs_reference.py."""
import numpy as np
import pytest

import assoc_ref
import restated_cases as rc
import scenes
from oracle import oracle_py as orc

pytestmark = pytest.mark.gpu

PRECS = [pytest.param(0, id="fp64"), pytest.param(1, id="tensor")]
TOLH = {0: 1e-9, 1: 1e-8}


@pytest.fixture(scope="module")
def gold():
    return rc.load()


def _pose_err(a, b):
    rot = max(np.linalg.norm(orc.log_so3(scenes.unpack_pose(x)[0].T @ scenes.unpack_pose(y)[0])) for x, y in zip(a, b))
    tra = max(np.linalg.norm(x[9:] - y[9:]) for x, y in zip(a, b))
    return rot, tra


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("n_poses,n_planes,drop,with_fix", rc.EVAL_SCENES)
def test_evaluators_match_the_stored_restatement(n_poses, n_planes, drop, with_fix, prec, gold):
    import balm_b200
    k = rc.EVAL_SCENES.index((n_poses, n_planes, drop, with_fix))
    sc = rc.eval_scene(n_poses, n_planes, drop, with_fix)
    coe = rc.coe_of(sc)
    o = orc.Oracle(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], coe, sc["fix10"])
    c = balm_b200.Context(n_poses, 0, prec)
    c.set_voxels(sc["row_ptr"], sc["pose_idx"], sc["obs10"], coe, sc["fix10"])
    for name in ("poses_init", "poses_gt"):
        x = sc[name]
        rr, gr, Hd = float(gold[f"eval{k}_{name}_r"]), gold[f"eval{k}_{name}_g"], gold[f"eval{k}_{name}_Hdiag"]
        H, g, r = c.evaluate(x)                              # (that evaluator ignores the fix cluster, bavoxel.hpp:325)
        assert abs(r - rr) <= 1e-10 * abs(rr), (r, rr)
        assert np.abs(g - gr).max() <= 1e-9 * np.abs(gr).max()
        assert np.abs(np.diag(H) - Hd).max() <= TOLH[prec] * np.abs(Hd).max()
        assert rc.probes_close(H, gold[f"eval{k}_{name}_Hprobes"], TOLH[prec])
        Ho, _, _ = o.evaluate_threads(x, threads=4)
        assert np.abs(H - Ho).max() <= TOLH[prec] * np.abs(Ho).max()
        assert abs(c.residual(x) - float(gold[f"eval{k}_{name}_residual"])) <= 1e-10 * abs(rr)   # fix cluster included
    lo, hi = rc.eval_range(n_planes)
    rr = float(gold[f"eval{k}_range_r"])
    H, g, r = c.evaluate(sc["poses_init"], lo, hi)
    assert abs(r - rr) <= 1e-10 * abs(rr)
    assert rc.probes_close(H, gold[f"eval{k}_range_Hprobes"], TOLH[prec])
    Ho, _, _ = o.evaluate(sc["poses_init"], lo, hi)
    assert np.abs(H - Ho).max() <= TOLH[prec] * np.abs(Ho).max()
    c.close()


@pytest.mark.parametrize("prec", PRECS)
def test_damping_iter_matches_the_stored_restatement(prec, gold):
    import balm_b200
    sc = rc.lm_scene()
    c = balm_b200.Context(24, 0, prec)
    c.set_voxels(sc["row_ptr"], sc["pose_idx"], sc["obs10"], rc.coe_of(sc))
    poses, tr, _ = c.damping_iter(sc["poses_init"], gauge_mode=0)
    assert len(tr) >= 3
    rot, tra = _pose_err(poses, gold["lm_poses"])            # the whole LM loop, gauge step included
    assert rot <= 1e-6 and tra <= 1e-6, (rot, tra)
    c.close()


def test_association_and_marginalisation_match_the_stored_restatement(gold):
    import balm_b200
    n, mg, kw = rc.ASSOC_N, rc.ASSOC_MG, rc.ASSOC_KW
    pts, frs, poses, poses12, opt = rc.assoc_inputs()
    keys, lay = gold["assoc_keys"], gold["assoc_layers"]     # cut_voxel per scan, recut, tras_opt -> push_voxel
    rp, pi, co = gold["assoc_row_ptr"], gold["assoc_pose_idx"], gold["assoc_coe"]
    c = balm_b200.Context(n, 0, 0)
    M, K = c.cut_voxels(pts.astype(np.float32), frs, poses12, **kw)
    kg, lg = c.download_keys(with_layers=True)
    rp_g, pi_g, ob_g, co_g = c.download_voxels()
    assert M == len(co) and K == len(pi) and M > 50
    assert np.array_equal(kg.astype(np.int64), keys) and np.array_equal(lg, lay)
    assert np.array_equal(rp_g, rp) and np.array_equal(pi_g, pi) and np.array_equal(co_g, co)
    _, _, ob, _, _ = assoc_ref.cut_voxels(pts, frs, poses, **kw)
    assert np.all(np.abs(ob_g - ob) <= 1e-11 * np.abs(ob).max(axis=0))
    assert rc.probes_close(ob_g, gold["assoc_obs_probes"], 1e-11)
    # retire the two oldest scans (OCTO_TREE_ROOT::marginalize on every root, consistency.cpp:131-135)
    rp1, pi1, co1 = gold["marg_row_ptr"], gold["marg_pose_idx"], gold["marg_coe"]
    _, _, ob1, fx1, _ = assoc_ref.marginalize_ref(n, rp, pi, ob, None, opt, mg, kw["min_ps"])
    M1, K1 = c.marginalize(mg, opt, min_ps=kw["min_ps"])
    rp_g, pi_g, ob_g, co_g = c.download_voxels()
    assert M1 == len(co1) and K1 == len(pi1)
    assert np.array_equal(c.download_keys().astype(np.int64), gold["marg_keys"])
    assert np.array_equal(rp_g, rp1) and np.array_equal(pi_g, pi1) and np.array_equal(co_g, co1)
    assert np.all(np.abs(ob_g - ob1) <= 1e-11 * np.abs(ob1).max(axis=0))
    assert rc.probes_close(ob_g, gold["marg_obs_probes"], 1e-11)
    fix = c.download_fix()
    assert np.abs(fix - fx1).max() <= 1e-12 * np.abs(fx1).max()
    assert rc.probes_close(fix, gold["marg_fix_probes"], 1e-12)
    c.close()
