"""The CUDA path against the REFERENCE'S OWN CODE, on the GPU box.

oracle/_ref/libbalm_ref.so -- the reference's src/benchmark/bavoxel.hpp + include/tools.hpp compiled where they lie behind
oracle/ref_harness.cpp (stand-ins for the absent Eigen / PCL / ROS headers, oracle/ref_stubs) -- is built where
BALM_REFERENCE_DIR names a checkout of the reference (tests/test_gpu_vs_restatement.py runs the same inputs elsewhere). Here the library's results (through the C ABI) are compared with
what the reference's own VOX_HESS / BALM2 / OCTO_TREE_ROOT produce on the same inputs: no restatement in between.
Tolerances as in tests/test_gpu_parity.py (SURVEY.md 8d)."""
import numpy as np
import pytest

import assoc_ref
import scenes
from oracle import oracle_py as orc
from oracle import ref_py as ref

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libbalm_ref.so not built (needs BALM_REFERENCE_DIR)")]

PRECS = [pytest.param(0, id="fp64"), pytest.param(1, id="tensor")]
TOLH = {0: 1e-9, 1: 1e-8}


def _pose_err(a, b):
    rot = max(np.linalg.norm(orc.log_so3(scenes.unpack_pose(x)[0].T @ scenes.unpack_pose(y)[0])) for x, y in zip(a, b))
    tra = max(np.linalg.norm(x[9:] - y[9:]) for x, y in zip(a, b))
    return rot, tra


def _coe(sc):  # the reference's push_voxel derives the weight itself: sum of N over the voxel (bavoxel.hpp:42-44)
    return np.array([sc["obs10"][a:b, 9].sum() for a, b in zip(sc["row_ptr"][:-1], sc["row_ptr"][1:])])


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("n_poses,n_planes,drop,with_fix", [(6, 40, 0.0, False), (37, 64, 0.0, False), (20, 200, 0.4, False),
                                                            (12, 50, 0.3, True)])
def test_evaluators_match_the_reference_code(n_poses, n_planes, drop, with_fix, prec):
    import balm_b200
    sc = scenes.make_scene(n_poses=n_poses, n_planes=n_planes, seed=31, drop=drop, with_fix=with_fix, pts_size=12)
    coe = _coe(sc)
    p = ref.Problem(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], sc["fix10"])
    assert p.pushed() == n_planes and np.array_equal(p.coeffs(), coe)
    c = balm_b200.Context(n_poses, 0, prec)
    c.set_voxels(sc["row_ptr"], sc["pose_idx"], sc["obs10"], coe, sc["fix10"])
    for x in (sc["poses_init"], sc["poses_gt"]):
        Hr, gr, rr = p.divide_thread_left(x)                 # BALM2::divide_thread_left: 4 x left_evaluate_acc2, ordered sum
        H, g, r = c.evaluate(x)                              # (that evaluator ignores the fix cluster, bavoxel.hpp:325)
        assert abs(r - rr) <= 1e-10 * abs(rr), (r, rr)
        assert np.abs(g - gr).max() <= 1e-9 * np.abs(gr).max()
        assert np.abs(H - Hr).max() <= TOLH[prec] * np.abs(Hr).max()
        assert abs(c.residual(x) - p.evaluate_only_residual(x)) <= 1e-10 * abs(rr)   # fix cluster included (:441)
    lo, hi = n_planes // 5, n_planes // 2                    # voxel range of one worker thread
    Hr, gr, rr = p.left_evaluate_acc2(sc["poses_init"], lo, hi)
    H, g, r = c.evaluate(sc["poses_init"], lo, hi)
    assert abs(r - rr) <= 1e-10 * abs(rr) and np.abs(H - Hr).max() <= TOLH[prec] * np.abs(Hr).max()
    c.close()


@pytest.mark.parametrize("prec", PRECS)
def test_damping_iter_matches_the_reference_code(prec):
    import balm_b200
    sc = scenes.make_scene(n_poses=24, n_planes=600, seed=18, pts_size=10)       # >= 20 planes per pose (bavoxel.hpp:1079)
    p = ref.Problem(24, sc["row_ptr"], sc["pose_idx"], sc["obs10"])
    poses_r = p.damping_iter(sc["poses_init"])               # BALM2::damping_iter: the whole loop, gauge step included
    c = balm_b200.Context(24, 0, prec)
    c.set_voxels(sc["row_ptr"], sc["pose_idx"], sc["obs10"], _coe(sc))
    poses, tr, _ = c.damping_iter(sc["poses_init"], gauge_mode=0)
    assert len(tr) >= 3
    rot, tra = _pose_err(poses, poses_r)
    assert rot <= 1e-6 and tra <= 1e-6, (rot, tra)           # north_star's bar; measured ~1e-9
    c.close()


def test_association_and_marginalisation_match_the_reference_octree():
    import balm_b200
    n, mg = 8, 2
    kw = dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 16))
    pts, frs, poses = assoc_ref.synthetic_scans(n_poses=n, pts_per_scan=4000, seed=22)
    poses12 = scenes.pack_poses([r for r, _ in poses], [p for _, p in poses])
    s = ref.Session(n, kw["voxel_size"], kw["layer_limit"], kw["min_ps"], kw["eigen_value_array"])
    for i in range(n):                                        # cut_voxel per scan, then recut (benchmark_realworld.cpp:187-197)
        s.cut_voxel(pts[frs == i].astype(np.float32), poses12[i], i)
    s.recut(n)
    keys, rp, pi, ob, fx, co, lay = s.export(n, with_layers=True)   # tras_opt -> push_voxel (:198)
    c = balm_b200.Context(n, 0, 0)
    M, K = c.cut_voxels(pts.astype(np.float32), frs, poses12, **kw)
    kg, lg = c.download_keys(with_layers=True)
    rp_g, pi_g, ob_g, co_g = c.download_voxels()
    assert M == len(co) and K == len(pi) and M > 50
    assert np.array_equal(kg.astype(np.int64), keys) and np.array_equal(lg, lay)
    assert np.array_equal(rp_g, rp) and np.array_equal(pi_g, pi) and np.array_equal(co_g, co)
    assert np.all(np.abs(ob_g - ob) <= 1e-11 * np.abs(ob).max(axis=0))
    # retire the two oldest scans: OCTO_TREE_ROOT::marginalize on every root (consistency.cpp:131-135) vs balm_marginalize
    rng = np.random.default_rng(1)
    opt = poses12.copy()
    opt[:, 9:] += rng.normal(0, 0.01, (n, 3))
    s.marginalize(mg, opt, n)
    keys1, rp1, pi1, ob1, fx1, co1 = s.export(n - mg)
    M1, K1 = c.marginalize(mg, opt, min_ps=kw["min_ps"])
    rp_g, pi_g, ob_g, co_g = c.download_voxels()
    assert M1 == len(co1) and K1 == len(pi1)
    assert np.array_equal(c.download_keys().astype(np.int64), keys1)
    assert np.array_equal(rp_g, rp1) and np.array_equal(pi_g, pi1) and np.array_equal(co_g, co1)
    assert np.all(np.abs(ob_g - ob1) <= 1e-11 * np.abs(ob1).max(axis=0))
    assert np.abs(c.download_fix() - fx1).max() <= 1e-12 * np.abs(fx1).max()
    c.close()
